"""GPU (B200): every policy against the CPU oracle on hand-built waveforms that sit at the edges the packed arithmetic relies on.

The synthetic generator (csrc/framegen.h) gives a constant pedestal, Gaussian noise and triangular pulses: its first sample is
never near a rail, its pedestal never moves, its pulses cross the threshold with a margin, its hits are short and its timestamps
step evenly. The cases below are built sample by sample instead (numpy, packed with frames.pack_wibeth_frames /
pack_wib2_superchunks, timestamp words written afterwards) and reach what the range arguments in swtpg_kernels.cuh are about:
quartile trackers seeded at a rail, pedestals that run from rail to rail, samples exactly at the threshold at every tick phase,
hits that saturate their time over threshold, equal peaks, collapsed quartiles, 32- and 64-bit timestamp edges, dead and stuck
channels.

Each case states the edge it reaches as a check on the oracle's outputs alone (`test_construction_reaches_its_edge`, no GPU
needed). The GPU tests run the same input through the library in one batch, in batches of one unit and in batches of an odd
length, and compare TPs, every state field the policy carries and the per-sample pedestal / waveform dumps with the oracle;
`test_constructed_cases_in_slices` reruns them with every launch handed out in 4 slices (SWTPG_PARTS=4)."""
import functools
import os
import subprocess
import sys
from dataclasses import dataclass, field

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B
from util import assert_same_state, assert_same_tps, channels, dump_states, ticks_per_unit

TS0 = 1 << 40
ANY_TAPS = [-3, 7, 20, 31, 20, 7, -3]  # test_gpu_parity.py ANY_TAPS[1]: PackedFirIqrAnyTaps

# policy -> (format, TPGenerator / oracle configuration). The acc_limit of the packed WIBEth policies may be overridden per case.
POLICIES = {
    "eth_simple": ("wibeth", dict(algorithm="SimpleThreshold", threshold=60)),
    "eth_absrs": ("wibeth", dict(algorithm="AbsRS", threshold=30)),
    "eth_stdrs": ("wibeth", dict(algorithm="StandardRS", threshold=30, rs_memory_factor=7, rs_scale_factor=2)),
    "eth_fir": ("wibeth", dict(algorithm="FIR", threshold=5)),                                    # binomial cascade, CTA form
    "eth_fir_any": ("wibeth", dict(algorithm="FIR", threshold=5, fir_taps=ANY_TAPS)),             # PackedFirIqrAnyTaps
    "eth_scalar": ("wibeth", dict(algorithm="SimpleThreshold", threshold=60, acc_limit=1001)),   # ScalarAlgo
    "wib2_simple": ("wib2", dict(algorithm="SimpleThreshold", threshold=64)),
    "wib2_fir": ("wib2", dict(algorithm="FIR", threshold=5)),
    "wib2_absrs": ("wib2", dict(algorithm="AbsRS", threshold=60)),
}
ETH = [p for p, (f, _) in POLICIES.items() if f == "wibeth"]
WIB2 = [p for p, (f, _) in POLICIES.items() if f == "wib2"]
ALL = ETH + WIB2
QUARTILES = ["eth_fir", "eth_fir_any", "wib2_fir", "wib2_absrs"]  # the policies that run PackedFirIqr::track()
WITH_ACC_LIMIT = ("eth_simple", "eth_absrs", "eth_stdrs")


# ---- builder ----------------------------------------------------------------------------------------------------------------
def pack_units(fmt, adc, ts):
    """adc [units][ticks][channels] (clipped to 14 bits), ts [units] -> the units' bytes. The timestamp words are written after
    packing, so consecutive units may have gaps and backward steps; the frames of a WIB2 superchunk are 32 apart (mod 2^64)."""
    adc = np.clip(adc, 0, 16383).astype(np.uint16)
    ts = np.asarray(ts, dtype=np.uint64)
    n = adc.shape[0]
    if fmt == "wibeth":
        u = F.pack_wibeth_frames(adc, 0)
        u[:, 8:16] = ts.astype("<u8").view(np.uint8).reshape(n, 8)
        return u
    u = F.pack_wib2_superchunks(adc.reshape(-1, F.WIB2_CHANNELS), 0).reshape(n, F.WIB2_SUPERCHUNK_FRAMES, F.WIB2_FRAME_BYTES)
    fts = ts[:, None] + np.uint64(F.TS_PER_TICK) * np.arange(F.WIB2_SUPERCHUNK_FRAMES, dtype=np.uint64)[None, :]
    words = np.stack([fts & np.uint64(0xFFFFFFFF), fts >> np.uint64(32)], axis=-1).astype("<u4")
    u[:, :, 4:12] = words.view(np.uint8).reshape(n, F.WIB2_SUPERCHUNK_FRAMES, 8)
    return u.reshape(n, F.WIB2_SUPERCHUNK_BYTES)


@dataclass
class Case:
    fmt: str
    sig: np.ndarray                  # [links][ticks][channels], a whole number of units
    ts: np.ndarray = None            # [units]; default: TS0 + ticks * 32, evenly
    kw: dict = field(default_factory=dict)  # configuration overrides
    odd: int = 7                     # units per batch of the odd-length batching
    unit_batches: bool = True        # also run in batches of one unit

    @property
    def n_units(self):
        return self.sig.shape[1] // ticks_per_unit(self.fmt)

    def timestamps(self):
        if self.ts is not None:
            return np.asarray(self.ts, dtype=np.uint64)
        return np.uint64(TS0) + np.uint64(ticks_per_unit(self.fmt) * F.TS_PER_TICK) * np.arange(self.n_units, dtype=np.uint64)

    def units(self):
        tpu = ticks_per_unit(self.fmt)
        return np.stack([pack_units(self.fmt, s.reshape(self.n_units, tpu, -1), self.timestamps()) for s in self.sig])


def ticks_for(fmt, n_ticks):
    """n_ticks rounded up to whole units."""
    tpu = ticks_per_unit(fmt)
    return -(-n_ticks // tpu) * tpu


# ---- the cases ------------------------------------------------------------------------------------------------------------
# Each builder takes the policy and returns a Case; the check next to it (CASES, POLICY_CHECKS) states on the oracle's outputs
# which edge the case reaches.
def case_rail_seed(policy):
    """1. Quartiles seeded at a rail: pedestal = first sample, q25 / q75 = it -+ 20 (ProcessingInfo.hpp:101-141). The first sample
    of a rail channel sweeps 16360..16383 over the lanes, so q75 starts at up to 16403; the channel then sits around 16300, the
    median comes down and q75 walks back through 16386 -> 16385 (the bias edge of the q75 register). Lanes 0-23 have the rail
    on the even channel and an ordinary odd neighbour, lanes 24-31 (mod 32) the other way round, with the ordinary even
    channel seeded at 0 (q25 = -20)."""
    fmt = POLICIES[policy][0]
    T, nch = ticks_for(fmt, 2560), channels(fmt)
    rng = np.random.default_rng(11)
    sig = np.zeros((1, T, nch), dtype=np.int32)
    for lane in range(nch // 2):
        j = lane % 32
        rail, other = (2 * lane, 2 * lane + 1) if j < 24 else (2 * lane + 1, 2 * lane)
        sig[0, :, rail] = 16300 + rng.integers(-3, 4, T)
        sig[0, 0, rail] = 16360 + j if j < 24 else 16376 + (j - 24)
        base = 500 if j < 24 else 300
        sig[0, :, other] = base + rng.integers(-3, 4, T)
        sig[0, 0, other] = base if j < 24 else 0
    return Case(fmt, sig)


def check_rail_seed(case, out):
    st = out["states"]  # [units][channels] after every unit
    q75 = st["quantile75"][:, 0::2]
    above = q75 >= 16386
    crossed = above.any(axis=0) & (q75[-1] <= 16385) & above[0]
    assert crossed.sum() >= 10, "too few even channels whose q75 went from 16386 or more to 16385 or less"
    seeded = np.nonzero(case.sig[0, 0] == 0)[0]
    assert seeded.size and (st["quantile25"][0, seeded] == -20).all(), "q25 of the channels seeded at 0 is not -20"
    assert (st["quantile75"][0] >= 16386).sum() >= 20, "q75 above 16385 on too few channels"


def case_moving(policy, L=None):
    """2. Moving pedestals: steps from rail to rail (0 -> 16383 -> 0), ramps of one count per tick, square waves; the two channels
    of a lane move in opposite directions, so both halves of a lane's accumulator register reach +-L on the same tick."""
    fmt = POLICIES[policy][0]
    T, nch = ticks_for(fmt, 2560), channels(fmt)
    t = np.arange(T)
    sig = np.zeros((1, T, nch), dtype=np.int32)
    for lane in range(nch // 2):
        kind = lane % 4
        if kind == 0:
            up = np.where((t // 320) % 2 == 1, 16383, 0)
        elif kind == 1:
            up = 2000 + t
        elif kind == 2:
            up = 8000 + np.where((t // 32) % 2 == 0, 1000, -1000)
        else:
            up = t * 7
        up = np.clip(up, 0, 16383)
        sig[0, :, 2 * lane] = up
        sig[0, :, 2 * lane + 1] = 16383 - up
    kw = {} if L is None else dict(acc_limit=L)
    return Case(fmt, sig, kw=kw)


def check_moving(case, out):
    ped = out["ped"][0].reshape(-1, case.sig.shape[2]).astype(np.int32)
    d = np.diff(ped, axis=0)
    opposite = ((d[:, 0::2] == 1) & (d[:, 1::2] == -1)) | ((d[:, 0::2] == -1) & (d[:, 1::2] == 1))
    assert opposite.any(), "no lane whose two pedestals step in opposite directions on the same tick"
    assert (ped == 0).any() and (ped == 16383).any(), "the pedestals do not reach both rails"


def exact_threshold_events(fmt, T):
    """(channel, first tick, kind) of every event of case_exact_threshold: kind 0 = s' == threshold for one tick, kind 1 = a
    one-tick hit at threshold + 1, one tick at -1, a second one-tick hit (ends on one tick, restarts on the next)."""
    tpu, nch = ticks_per_unit(fmt), channels(fmt)
    offs = (-1, 0, 1, 2, 3, 31, 32) if fmt == "wibeth" else (-1, 0, 1, 2, 3, 5, 6)
    ev = []
    for c in range(nch):
        for f in range(1, T // tpu - 1):
            ev.append((c, f * tpu + offs[(c + f) % len(offs)], 0 if (c + f) % 3 == 0 else 1))
    return ev


def case_exact_threshold(policy):
    """3. Samples exactly at the threshold: s' = threshold (no hit) and threshold + 1 (a one-tick hit), at every tick phase mod 4
    (the quiet test's group), around tick 31/32 (the ring chunk) and 63/0 (frame) of WIBEth, 11/0 of WIB2, and so at batch and
    slice edges too, on even and odd channels. Every excursion above the pedestal is paid back by one tick at -1, so the median
    never moves and s' is exact."""
    fmt, cfg = POLICIES[policy]
    thr = cfg["threshold"]
    T, nch, P = ticks_for(fmt, 1280), channels(fmt), 1000
    sig = np.full((1, T, nch), P, dtype=np.int32)
    for c, t0, kind in exact_threshold_events(fmt, T):
        seq = [thr, -1] if kind == 0 else [thr + 1, -1, thr + 1, -1]
        sig[0, t0:t0 + len(seq), c] = P + np.array(seq)
    return Case(fmt, sig)


def check_exact_threshold(case, out):
    fmt = case.fmt
    thr = POLICIES["wib2_simple" if fmt == "wib2" else "eth_simple"][1]["threshold"]
    ev = exact_threshold_events(fmt, case.sig.shape[1])
    tps = out["tps"][0]
    assert (out["ped"][0] == 1000).all(), "the pedestal moved: s' is not exact"
    assert tps.size == 2 * sum(k for _, _, k in ev), "not one TP per sample above the threshold"
    assert (tps["time_over_threshold"] == F.TS_PER_TICK).all()
    if fmt == "wibeth":
        assert (tps["adc_integral"] == thr + 1).all() and (tps["adc_peak"] == thr + 1).all()
    starts = {(c, t0) for c, t0, k in ev if k}
    got = {(int(tp["channel"]), int((int(tp["time_start"]) - TS0) // F.TS_PER_TICK)) for tp in tps}
    assert starts <= got and {(c, t0 + 2) for c, t0 in starts} <= got, "a one-tick hit at threshold + 1 is missing"
    phases = {t0 % ticks_per_unit(fmt) for _, t0, k in ev if k}
    assert {0, 1, 2, 3, ticks_per_unit(fmt) - 1} <= phases
    assert {c % 2 for c, _, k in ev if k} == {0, 1}


LONG_TICKS = 38400  # > 32767: the time over threshold saturates


def case_long_hit(policy):
    """4. Long hits: a channel seeded at 0 jumps to 16383 for 38400 ticks (600 WIBEth frames, 3200 WIB2 superchunks) and back.
    The pedestal needs about 180 k ticks to catch up at L = 10, so the hit stays open across every batch and slice boundary of
    the run and its time over threshold saturates at 32767; the charge of the running sums and of WIB2 saturates at 32767.
    Two such channels (even and odd), one starting 5 ticks late; the other channels sit at a constant 500."""
    fmt = POLICIES[policy][0]
    T, nch = ticks_for(fmt, LONG_TICKS + 600), channels(fmt)
    sig = np.full((1, T, nch), 500, dtype=np.int32)
    for c, t0 in ((0, 1), (3, 6)):
        sig[0, :, c] = 0
        sig[0, t0:t0 + LONG_TICKS, c] = 16383
    return Case(fmt, sig, odd=37 if fmt == "wibeth" else 97, unit_batches=False)


def check_long_hit(case, out, policy):
    tps = out["tps"][0]
    tps = tps[np.isin(tps["channel"], (0, 3))]
    assert tps.size, "no TP on the long-hit channels"
    if policy == "eth_fir_any":  # taps summing to 79: 79 * adcMax wraps to a negative filter output, so the step is no hit
        assert (out["wav"][0][..., 0] == np.int16(79 * 511 - 65536)).sum() > 30000, "the filter output does not wrap"
    elif policy in ("eth_absrs", "eth_stdrs", "wib2_absrs"):
        assert (tps["adc_integral"] == 32767).any(), "no saturated charge"
    else:
        assert (tps["time_over_threshold"] == 32767 * F.TS_PER_TICK).any(), "no saturated time over threshold"


def case_charge_wrap(policy):
    """4b. WIBEth SimpleThreshold adds the charge modulo 2^16 (H3): a 5-tick hit whose s' sums to exactly 65536 ends with charge 0,
    so it is not a TP (WIBEthFrameProcessor.cpp:520-545) and its state is reset; the next hit on the channel is an ordinary TP.
    s' = 13107 x 4 + 13108 on a flat pedestal of 100, paid back by 5 ticks at -1 so the median does not move."""
    fmt = POLICIES[policy][0]
    T, nch, P = ticks_for(fmt, 640), channels(fmt), 100
    sig = np.full((1, T, nch), P, dtype=np.int32)
    for c in range(nch):
        t0 = 70 + 3 * c
        sig[0, t0:t0 + 10, c] = P + np.array([13107] * 4 + [13108] + [-1] * 5)
        sig[0, t0 + 200:t0 + 204, c] = P + np.array([300, 400, -1, -1])
    return Case(fmt, sig)


def check_charge_wrap(case, out):
    tps = out["tps"][0]
    assert tps.size == case.sig.shape[2], "expected exactly the one ordinary hit per channel"
    assert (tps["adc_integral"] == 300 + 400).all() and (tps["adc_peak"] == 400).all()
    assert (out["ped"][0] == 100).all()


def case_peaks(policy):
    """5. Peaks: a hit with two equal maxima (the first one is the peak: `x > peak`, ProcessAVX2.hpp:134-136) and, for the running
    sums, a quiet tick whose s' is larger than any sample of the following hit: the peak tracker is not gated by the hit (H6), so
    that quiet tick is the hit's peak. A last quiet spike leaves its value in the carried peak state."""
    fmt, cfg = POLICIES[policy]
    T, nch, P = ticks_for(fmt, 1280), channels(fmt), 1000
    spike, level = {"eth_absrs": (55, 40), "eth_stdrs": (250, 200)}.get(policy, (cfg["threshold"], 0))
    sig = np.full((1, T, nch), P, dtype=np.int32)
    for c in range(nch):
        t0 = 70 + 5 * c
        sig[0, t0:t0 + 10, c] = P + np.array([300, 600, 450, 600, 300] + [-1] * 5)
        if level:
            sig[0, t0 + 200:t0 + 202, c] = P + np.array([spike, -1])
            sig[0, t0 + 240:t0 + 252, c] = P + np.array([level] * 6 + [-1] * 6)
        sig[0, T - 20:T - 18, c] = P + np.array([cfg["threshold"], -1])
    return Case(fmt, sig)


def check_peaks(case, out, policy):
    tps = out["tps"][0]
    first_max = TS0 + F.TS_PER_TICK * (70 + 5 * tps["channel"].astype(np.uint64) + 1)
    big = tps["adc_peak"] == 600
    assert big.sum() == case.sig.shape[2] and (tps["time_peak"][big] == first_max[big]).all(), "equal maxima: not the first one"
    if policy in ("eth_absrs", "eth_stdrs"):
        spike = {"eth_absrs": 55, "eth_stdrs": 250}[policy]
        q = tps[tps["adc_peak"] == spike]
        assert q.size == case.sig.shape[2] and (q["time_peak"] == q["time_start"]).all(), "no peak taken from a quiet tick"
    assert (out["final"]["hit_peak_adc"] == POLICIES[policy][1]["threshold"]).all(), "the last quiet spike is not the carried peak"


def case_narrow_iqr(policy, one_lane=False):
    """6. Collapsed quartiles: samples alternating median + 1 / median - 1 pull q75 and q25 to within 2 of the median (sigma 2),
    then samples equal to the median freeze every tracker. With sigma < 3 the quiet test's lower bound of the group's sigmas is
    negative, so every group is busy and the per-tick thresholds are formed; sigma * multiplier * threshold is then below the
    filter output of a small pulse. In the one-lane variant only lane 5 (channels 10, 11) of each 64 channels collapses; the
    others keep q25 / q75 = pedestal -+ 20."""
    fmt = POLICIES[policy][0]
    T, nch, P = ticks_for(fmt, 1920), channels(fmt), 1000
    t = np.arange(T)
    sig = np.full((1, T, nch), P, dtype=np.int32)
    narrow = [c for c in range(nch) if not one_lane or c % 64 in (10, 11)]
    for c in narrow:
        sig[0, 1:1200, c] = P + np.where(t[1:1200] % 2 == 0, 1, -1)
    for c in range(3, nch, 8):
        sig[0, 1400 + c % 40:1404 + c % 40, c] = P + np.array([400, 600, 400, 200])
    return Case(fmt, sig)


def check_narrow_iqr(case, out, one_lane=False):
    st = out["final"]
    sigma = st["quantile75"].astype(int) - st["quantile25"]
    nch = sigma.size
    narrow = np.array([not one_lane or c % 64 in (10, 11) for c in range(nch)])
    assert (sigma[narrow] <= 2).all() and (sigma[narrow] >= 0).all(), sigma[narrow]
    assert (sigma[~narrow] == 40).all()
    assert out["tps"][0].size > 0


def ts_edges(fmt, n_units):
    """Per-unit timestamps of case_timestamps: WIBEth units 0-4 end just under a 2^32 boundary (unit 5 starts on it); WIB2 runs
    within 2^20 of 2^64 (t_begin + t_stop overflows 64 bits). Both: a gap of 100 units after unit 5, a step back of 50 after
    unit 6."""
    step = ticks_per_unit(fmt) * F.TS_PER_TICK
    base = (7 << 32) - 5 * step if fmt == "wibeth" else (1 << 64) - 200 * step - 1000
    ts = []
    for u in range(n_units):
        t = base + u * step
        if u >= 6:
            t += 99 * step
        if u >= 7:
            t -= 51 * step
        ts.append(t % (1 << 64))
    return np.array(ts, dtype=np.uint64)


def case_timestamps(policy):
    """7. Timestamps: hits open across the unit boundaries 4|5 (2^32 carry of WIBEth's time_start, which borrows across 32 bits),
    5|6 (a forward gap) and 6|7 (a backward step): the TP takes the timestamp of the unit where it ends. WIB2 near 2^64."""
    fmt = POLICIES[policy][0]
    tpu, nch, P = ticks_per_unit(fmt), channels(fmt), 1000
    n_units = 12
    T = n_units * tpu
    sig = np.full((1, T, nch), P, dtype=np.int32)
    for c in range(nch):
        b = (5 + c % 3) * tpu - 4 * (c % 2)  # odd channels 4 ticks early: the FIR output lags the samples
        w = 3 if fmt == "wib2" else 4 + c % 4
        sig[0, b - w:b + w, c] = P + 600
        sig[0, b + w:b + 3 * w, c] = P - 1
    return Case(fmt, sig, ts=ts_edges(fmt, n_units))


def check_timestamps(case, out):
    tps = out["tps"][0]
    assert tps.size > 0
    ts = case.timestamps()
    end = tps["time_start"] + tps["time_over_threshold"].astype(np.uint64)  # wraps like the reference's uint64
    if case.fmt == "wibeth":
        assert ((tps["time_start"] >> np.uint64(32)) == 6).any() and ((end >> np.uint64(32)) == 7).any(), "no 2^32 borrow"
    else:
        assert (tps["time_peak"] < tps["time_start"]).any(), "t_begin + t_stop never overflows"
    # a TP ending in unit 6 (after the gap) or 7 (after the step back) that started in the unit before is stamped from the
    # timestamp of the unit where it ends: it starts less than one unit before that timestamp
    span = ts.dtype.type(ticks_per_unit(case.fmt) * F.TS_PER_TICK)
    assert any(((tps["time_start"] < ts[u]) & (tps["time_start"] > ts[u] - span)).any() for u in (6, 7)), "no hit across the gap"


def case_dead_stuck(policy):
    """8. Dead and stuck channels: one in four held at 0, one at 16383, one alternating 0 / 16383 on every tick, one ordinary
    with pulses."""
    fmt = POLICIES[policy][0]
    T, nch = ticks_for(fmt, 1024), channels(fmt)
    t = np.arange(T)
    rng = np.random.default_rng(8)
    sig = np.zeros((1, T, nch), dtype=np.int32)
    sig[0, :, 1::4] = 16383
    sig[0, :, 2::4] = np.where(t % 2, 16383, 0)[:, None]
    sig[0, :, 3::4] = 800 + rng.integers(-4, 5, (T, nch // 4))
    for k in range(1, 8):
        sig[0, 128 * k:128 * k + 6, 3::4] += 500
    return Case(fmt, sig)


def check_dead_stuck(case, out):
    ped = out["final"]["pedestal"]
    assert (ped[0::4] == 0).all() and (ped[1::4] == 16383).all()
    alt = out["ped"][0][..., 2::4]
    assert alt.min() == 0 and alt.max() <= 2, "the alternating channels' pedestal should stay at the low rail"
    assert out["tps"][0].size > 0


CASES = {
    # name: (builder, policies, check)
    "rail_seed": (case_rail_seed, QUARTILES, check_rail_seed),
    "moving_L1": (functools.partial(case_moving, L=1), WITH_ACC_LIMIT, check_moving),
    "moving_L1000": (functools.partial(case_moving, L=1000), WITH_ACC_LIMIT, check_moving),
    "moving": (case_moving, ["eth_scalar", "eth_fir", "eth_fir_any"] + WIB2, check_moving),
    "exact_threshold": (case_exact_threshold, ["eth_simple", "eth_scalar", "wib2_simple"], check_exact_threshold),
    "long_hit": (case_long_hit, ALL, None),
    "charge_wrap": (case_charge_wrap, ["eth_simple", "eth_scalar"], check_charge_wrap),
    "peaks": (case_peaks, ["eth_simple", "eth_absrs", "eth_stdrs", "eth_scalar"], None),
    "narrow_iqr": (case_narrow_iqr, QUARTILES, check_narrow_iqr),
    "narrow_iqr_one_lane": (functools.partial(case_narrow_iqr, one_lane=True), QUARTILES,
                            functools.partial(check_narrow_iqr, one_lane=True)),
    "timestamps": (case_timestamps, ALL, check_timestamps),
    "dead_stuck": (case_dead_stuck, ALL, check_dead_stuck),
}
POLICY_CHECKS = {"long_hit": check_long_hit, "peaks": check_peaks}
PAIRS = [(c, p) for c, (_, pols, _) in CASES.items() for p in pols]


# ---- oracle and comparison ------------------------------------------------------------------------------------------------
def config_of(case, policy):
    kw = dict(POLICIES[policy][1])
    if policy in WITH_ACC_LIMIT:
        kw.update(case.kw)
    return kw


@functools.lru_cache(maxsize=None)
def build(name, policy):
    return CASES[name][0](policy)


@functools.lru_cache(maxsize=None)
def oracle_run(name, policy):
    """The oracle over the whole case, one link at a time: TPs, pedestal and waveform dumps, final state; and the state after
    every unit (link 0) for the checks that read it between units."""
    case = build(name, policy)
    kw = config_of(case, policy)
    algorithm = kw.pop("algorithm")
    units = case.units()
    cfg = B.make_config(fmt=case.fmt, algorithm=S.ALGORITHMS[algorithm], **kw)
    tps, peds, wavs, finals = [], [], [], []
    states = None
    for l in range(units.shape[0]):
        o = B.Oracle(cfg, link_id=l)
        if name == "rail_seed" and l == 0:
            parts, ps, ws, states = [], [], [], []
            for u in range(units.shape[1]):
                t, p, w = o.process(units[l, u:u + 1], dump=True, cap=1 << 20)
                parts.append(t), ps.append(p), ws.append(w), states.append(o.state())
            t, p, w = np.concatenate(parts), np.concatenate(ps), np.concatenate(ws)
            states = np.stack(states)
        else:
            t, p, w = o.process(units[l], dump=True, cap=1 << 20)
        tps.append(t), peds.append(p), wavs.append(w), finals.append(o.state())
    return dict(units=units, tps=tps, ped=np.stack(peds), wav=np.stack(wavs), final=finals[0], finals=np.stack(finals), states=states)


def run_gpu(name, policy, step, sorted_tps=False):
    case = build(name, policy)
    want = oracle_run(name, policy)
    units = want["units"]
    n_links, n = units.shape[0], units.shape[1]
    got, gp, gw = [], [], []
    with S.TPGenerator(n_links, step, fmt=case.fmt, tp_capacity=1 << 21, sorted_tps=sorted_tps, **config_of(case, policy)) as g:
        g.start()
        for u in range(0, n, step):
            chunk = np.ascontiguousarray(units[:, u:u + step])
            t, p, w = g.process_host(chunk, units_stride=chunk.shape[1], debug=True, cap=1 << 21)
            got.append(t), gp.append(p), gw.append(w)
        states = dump_states(g)
    return got, np.concatenate(gp, axis=1), np.concatenate(gw, axis=1), states


def compare(name, policy, step):
    want = oracle_run(name, policy)
    got, gp, gw, gstate = run_gpu(name, policy, step)
    what = f"{name} / {policy} / {step} units per batch"
    assert_same_tps(np.concatenate(got), np.concatenate(want["tps"]), what)
    fmt, cfg = POLICIES[policy]
    assert_same_state(gstate, want["finals"], fmt, cfg["algorithm"], what)
    for label, g, w in (("pedestal", gp, want["ped"]), ("waveform", gw, want["wav"])):
        bad = g != w
        if bad.any():
            l, u, t, c = (int(i[0]) for i in np.nonzero(bad))
            pytest.fail(f"{what}: {label} dump differs at {int(bad.sum())} samples, first link {l} unit {u} tick {t} channel {c}: "
                        f"GPU {g[l, u, t, c]}, oracle {w[l, u, t, c]}")
    return got


def batchings(name, policy):
    case = build(name, policy)
    out = [("whole", case.n_units), ("odd", case.odd)]
    if case.unit_batches:
        out.append(("unit", 1))
    return out


# ---- CPU: every construction reaches its edge on the oracle ---------------------------------------------------------------
@pytest.mark.parametrize("name,policy", PAIRS, ids=[f"{c}-{p}" for c, p in PAIRS])
def test_construction_reaches_its_edge(name, policy):
    case = build(name, policy)
    out = oracle_run(name, policy)
    assert out["ped"].shape[1] == case.n_units
    if name in POLICY_CHECKS:
        POLICY_CHECKS[name](case, out, policy)
    else:
        CASES[name][2](case, out)


def test_builder_round_trip():
    """The builder's frames unpack to the samples and timestamps it was given (WIB2: every frame of a superchunk 32 later)."""
    rng = np.random.default_rng(3)
    adc = rng.integers(0, 16384, (3, 64, 64))
    ts = np.array([(1 << 32) - 2048, 5, (1 << 64) - 1], dtype=np.uint64)
    a, t = F.unpack_wibeth_frames(pack_units("wibeth", adc, ts))
    assert (a == adc).all() and (t == ts).all()
    adc2 = rng.integers(0, 16384, (2, 12, 256))
    ts2 = np.array([(1 << 64) - 100, 7], dtype=np.uint64)
    a2, t2 = F.unpack_wib2_superchunks(pack_units("wib2", adc2, ts2))
    assert (a2 == adc2.reshape(-1, 256)).all()
    assert (t2 == (ts2[:, None] + np.uint64(32) * np.arange(12, dtype=np.uint64)).reshape(-1)).all()


# ---- GPU: the library against the oracle ----------------------------------------------------------------------------------
GPU_PARAMS = [(c, p, b, s) for c, p in PAIRS for b, s in batchings(c, p)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,policy,batching,step", GPU_PARAMS, ids=[f"{c}-{p}-{b}" for c, p, b, _ in GPU_PARAMS])
def test_gpu_equals_oracle(name, policy, batching, step):
    compare(name, policy, step)


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ALL)
def test_gpu_device_ordered_timestamps(policy):
    """The timestamp edges with SWTPG_FLAG_SORTED_TPS: each batch's list comes back in the host order of its unordered list."""
    step = build("timestamps", policy).odd
    plain, _, _, _ = run_gpu("timestamps", policy, step)
    ordered, _, _, _ = run_gpu("timestamps", policy, step, sorted_tps=True)
    assert sum(p.size for p in plain) > 0
    for a, b in zip(ordered, plain):
        want = S.sort_tps(b)
        assert a.size == want.size and (a == want).all()


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("SWTPG_PARTS") is not None, reason="already running with forced slicing")
def test_constructed_cases_in_slices():
    """Every GPU case above with every launch handed out in 4 slices (SWTPG_PARTS=4): open hits, tracker steps and the FIR ring
    cross slice boundaries inside a batch as well."""
    env = dict(os.environ, SWTPG_PARTS="4")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "test_gpu_equals_oracle and not unit", "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, cwd=root)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout, r.stdout[-2000:]

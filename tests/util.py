"""Shared test code: bit-exact comparisons with the oracle and the reference, the carried-state rule, and the harness of the GPU
test modules (device and host-batch runners, the oracle replays, the launch rules restated)."""
import ctypes as C
import hashlib
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import api as A
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B

FIELDS = ("time_start", "time_peak", "time_over_threshold", "adc_integral", "adc_peak", "channel", "link")


def channels(fmt):
    return F.WIB2_CHANNELS if fmt == "wib2" else F.WIBETH_CHANNELS


def unit_bytes(fmt):
    return F.WIB2_SUPERCHUNK_BYTES if fmt == "wib2" else F.WIBETH_FRAME_BYTES


def ticks_per_unit(fmt):
    return F.WIB2_SUPERCHUNK_FRAMES if fmt == "wib2" else F.WIBETH_TICKS


# ---- comparisons ----------------------------------------------------------------------------------------------------------
def assert_same_tps(got: np.ndarray, want: np.ndarray, what: str = ""):
    """Bit-exact comparison of two TP lists as sorted field tuples."""
    g, w = F.sort_tps(np.asarray(got, dtype=F.TP_DTYPE)), F.sort_tps(np.asarray(want, dtype=F.TP_DTYPE))
    assert g.size == w.size, f"{what}: {g.size} TPs, expected {w.size}"
    for f in FIELDS:
        bad = np.nonzero(g[f] != w[f])[0]
        assert bad.size == 0, f"{what}: field {f} differs at sorted index {bad[0]}: got {g[bad[0]]}, want {w[bad[0]]}"


def digest(name: str, a: np.ndarray) -> np.ndarray:
    """SHA-256 of an output array, a TP list in canonical order."""
    if name == "tps":
        a = F.sort_tps(np.asarray(a, dtype=F.TP_DTYPE))
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def assert_same_as_reference(got: dict, ref, key: str):
    """got: {name: array} for the input `key` of tests/cases.py:reference_runs; ref: tests/golden/reference_outputs.npz, which
    holds each array either as it is ("<key>__<name>") or, when it is large, as its length and digest."""
    for name, a in got.items():
        k = f"{key}__{name}"
        if k in ref.files:
            if name == "tps":
                assert_same_tps(a, ref[k], key)
            else:
                assert a.shape == ref[k].shape and (a == ref[k]).all(), f"{key}: {name} differs from the reference"
        else:
            assert a.size == ref[k + "_count"][0], f"{key}: {a.size} {name}, the reference has {ref[k + '_count'][0]}"
            assert (digest(name, a) == ref[k + "_sha256"]).all(), f"{key}: {name} differs from the reference (digest)"


def oracle_config(case, B):
    return B.make_config(fmt=case["fmt"], algorithm=S.ALGORITHMS[case["algorithm"]], threshold=case["threshold"],
                         acc_limit=case.get("acc_limit", 10), rs_memory_factor=case.get("rs_memory_factor", 8),
                         rs_scale_factor=case.get("rs_scale_factor", 5))


# ---- carried state ----------------------------------------------------------------------------------------------------------
def state_fields(fmt, algorithm):
    """The fields of frames.STATE_DTYPE that a link of this format and algorithm carries from unit to unit; the others keep
    their seeds. tests/test_oracle_golden.py::test_state_fields_cover_what_moves checks the rule against the oracle."""
    f = ["pedestal", "accum", "prev_was_over", "hit_charge", "hit_tover", "initialized"]
    if fmt == "wibeth" and algorithm != "FIR":
        f += ["hit_peak_adc", "hit_peak_time"]
    if algorithm in ("AbsRS", "StandardRS"):
        f += ["rs", "pedestal_rs", "accum_rs"]
        if fmt == "wibeth":
            f += ["rs_memory_factor"]
    if algorithm == "FIR" or (fmt, algorithm) == ("wib2", "AbsRS"):  # WIB2 AbsRS tracks the quartiles of its sigma
        f += ["quantile25", "quantile75", "accum25", "accum75"]
    if algorithm == "FIR":
        f += ["prev_samp"]
    return f


def dump_states(g):
    """[links][channels] carried state of a TPGenerator."""
    return np.stack([g.dump_state(l) for l in range(g.n_links)])


def assert_same_state(gstate, ostate, fmt, algorithm, what):
    """Carried state [links][channels] against the oracle's on the fields state_fields names for each link's algorithm
    (`algorithm`: one for every link, or a function of the link). Reports the first differing link and channel."""
    of = algorithm if callable(algorithm) else (lambda l: algorithm)
    algos = np.array([of(l) for l in range(gstate.shape[0])])
    for a in np.unique(algos):
        links = np.nonzero(algos == a)[0]
        for f in state_fields(fmt, a):
            g, o = gstate[f][links], ostate[f][links]
            bad = (g != o).reshape(len(links), gstate.shape[1], -1).any(axis=2)
            if bad.any():
                i, ch = (int(x[0]) for x in np.nonzero(bad))
                pytest.fail(f"{what}: {a} state field {f} differs on {int(bad.any(axis=1).sum())} links, first link {int(links[i])} "
                            f"channel {ch}: GPU {g[i][ch]}, oracle {o[i][ch]}")


# ---- ADC statistics ---------------------------------------------------------------------------------------------------------
def adc_of(fmt, units, adc_offset=F.WIB2_ADC_OFFSET):
    """(samples, channels) raw ADC values of a link's units."""
    if len(units) == 0:
        return np.zeros((0, channels(fmt)), dtype=np.uint16)
    if fmt == "wib2":
        return F.unpack_wib2_superchunks(units, adc_offset)[0].reshape(-1, F.WIB2_CHANNELS)
    return F.unpack_wibeth_frames(units)[0].reshape(-1, F.WIBETH_CHANNELS)


def stats_of(a):
    """ADC_STATS_DTYPE row of (samples, channels) ADC values."""
    out = np.zeros(a.shape[1], dtype=F.ADC_STATS_DTYPE)
    if a.shape[0]:
        v = a.astype(np.uint64)
        out["samples"] = a.shape[0]
        out["sum"] = v.sum(0)
        out["sum_sq"] = (v * v).sum(0)
        out["min"] = a.min(0)
        out["max"] = a.max(0)
    return out


def expected(fmt, frames, nu=None, adc_offset=F.WIB2_ADC_OFFSET):
    """(n_links, channels) statistics of one batch: frames [n_links, stride, unit_bytes], nu valid units per link (None = all)."""
    n, stride = frames.shape[:2]
    return np.stack([stats_of(adc_of(fmt, frames[l, : (stride if nu is None else int(nu[l]))], adc_offset)) for l in range(n)])


def combine(a, b):
    """Statistics of two windows together."""
    out = a.copy()
    for f in ("samples", "sum", "sum_sq"):
        out[f] = a[f] + b[f]
    both = (a["samples"] > 0) & (b["samples"] > 0)
    out["min"] = np.where(both, np.minimum(a["min"], b["min"]), np.where(a["samples"] > 0, a["min"], b["min"]))
    out["max"] = np.maximum(a["max"], b["max"])
    return out


def ragged_batch(fmt, seed, n_links, stride, nu, **gen_kw):
    """Generated frames with every byte past each link's n_units set to 0xFF (an overread would count 16383s)."""
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    frames = gen(S.gen_params(seed, 0.3), n_links, stride, unit0=seed * stride, **gen_kw).copy()
    for l in range(n_links):
        frames[l, int(nu[l]):] = 0xFF
    return frames


# ---- noise lags -------------------------------------------------------------------------------------------------------------
def lags_of(fmt, a):
    """NOISE_LAGS_DTYPE row of (samples, channels) ADC values of one link in one batch: whole segments from the first sample."""
    n = F.NOISE_SEGMENT_TICKS[fmt]
    out = np.zeros(a.shape[1], dtype=F.NOISE_LAGS_DTYPE)
    segs = a.shape[0] // n
    x = a[: segs * n].astype(np.int64).reshape(segs, n, a.shape[1])
    out["segments"] = segs
    for tau in range(n // 2 + 1):
        out["lag"][:, tau] = (x * np.roll(x, -tau, axis=1)).sum(axis=(0, 1))
    return out


def expected_lags(fmt, frames, nu=None, adc_offset=F.WIB2_ADC_OFFSET):
    """(n_links, channels) lags of one batch: frames [n_links, stride, unit_bytes], nu valid units per link (None = all)."""
    n, stride = frames.shape[:2]
    return np.stack([lags_of(fmt, adc_of(fmt, frames[l, : (stride if nu is None else int(nu[l]))], adc_offset)) for l in range(n)])


# ---- channel products -------------------------------------------------------------------------------------------------------
def words_of(fmt, a):
    """One link's swtpg_read_channel_products row of (samples, channels) ADC values."""
    c = channels(fmt)
    x = np.asarray(a, dtype=np.int64).reshape(-1, c)
    out = np.zeros(F.channel_products_words(fmt), dtype=np.uint64)
    out[0] = x.shape[0]
    out[1:1 + c] = x.sum(axis=0)
    i, j = np.triu_indices(c)
    out[1 + c:] = (x.T @ x)[i, j]  # below 2^63 for every window of these tests: ticks x 16383^2
    return out


def expected_products(fmt, frames, nu=None, adc_offset=F.WIB2_ADC_OFFSET):
    """(n_links, words) of one batch: frames [n_links, stride, unit_bytes], nu valid units per link (None = all)."""
    n, stride = frames.shape[:2]
    return np.stack([words_of(fmt, adc_of(fmt, frames[l, : (stride if nu is None else int(nu[l]))], adc_offset)) for l in range(n)])


# ---- configurations ---------------------------------------------------------------------------------------------------------
# what TPGenerator's own configuration defaults to
HANDLE = dict(algorithm="SimpleThreshold", threshold=60, acc_limit=10, rs_memory_factor=8, rs_scale_factor=5, fir_taps=None, tap_exponent=6)
TPG_KEYS = tuple(HANDLE)


def full_conf(handle, link_kw):
    """The configuration of a link: the handle's keyword arguments over HANDLE, its set_link_config ones over those."""
    return {**HANDLE, **{k: v for k, v in handle.items() if k in TPG_KEYS}, **link_kw}


def oracle_for(fmt, conf, link):
    cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS[conf["algorithm"]], threshold=conf["threshold"], acc_limit=conf["acc_limit"],
                        rs_memory_factor=conf["rs_memory_factor"], rs_scale_factor=conf["rs_scale_factor"], fir_taps=conf["fir_taps"],
                        tap_exponent=conf["tap_exponent"])
    return B.Oracle(cfg, link_id=link)


def configured_oracles(fmt, handle, link_kw=None, rs_tables=None):
    """oracle_of(link) for links configured by link_kw {link: set_link_config kwargs} and rs_tables {link: per-channel RS memory
    factors}."""
    def oracle_of(l):
        o = oracle_for(fmt, full_conf(handle, (link_kw or {}).get(l, {})), l)
        if rs_tables is not None and l in rs_tables:
            o.set_memory_factor(rs_tables[l])
        return o

    return oracle_of


def all_wibeth_policies():
    any_taps = list(S.firwin_int(7, 0.1, 32))
    return [dict(algorithm="SimpleThreshold", threshold=30),
            dict(algorithm="AbsRS", threshold=30, rs_memory_factor=7, rs_scale_factor=2),
            dict(algorithm="StandardRS", threshold=30, rs_memory_factor=6),
            dict(algorithm="FIR", threshold=5),
            dict(algorithm="FIR", threshold=5, fir_taps=any_taps),  # not the binomial taps: PackedFirIqrAnyTaps
            dict(algorithm="SimpleThreshold", threshold=30, acc_limit=0)]  # the scalar fallback


def link_config(**kw):
    """A swtpg_link_config for the C ABI: SimpleThreshold at 60, accumulator limit 10, RS factors 8 / 5, fields set by kw."""
    c = _lib.SwtpgLinkConfig()
    c.struct_size = C.sizeof(c)
    c.algorithm, c.threshold, c.frugal_acc_limit, c.rs_memory_factor, c.rs_scale_factor = 0, 60, 10, 8, 5
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def create_status(fmt="wibeth", algorithm="SimpleThreshold", threshold=60, flags=0):
    """swtpg_create's status for a small handle: the configuration's error, else SWTPG_OK on a GPU and SWTPG_ERR_CUDA without
    one (the configuration is checked before any device is touched)."""
    cfg = _lib.SwtpgConfig()
    cfg.struct_size = C.sizeof(cfg)
    cfg.format, cfg.algorithm = A.FORMATS[fmt], S.ALGORITHMS[algorithm]
    cfg.n_links, cfg.max_units, cfg.threshold, cfg.frugal_acc_limit = 2, 4, threshold, 10
    cfg.flags = flags
    h = C.c_void_p()
    st = _lib.lib.swtpg_create(C.byref(cfg), C.byref(h))
    if h:
        _lib.lib.swtpg_destroy(h)
    return st


# ---- GPU harness --------------------------------------------------------------------------------------------------------------
# SWTPG_PARTS (the forced-slicing test hook) changes the geometry a launch takes: under it the regimes the launch-geometry and
# per-link tests assert are not the ones that run.
TUNING_AIDS = ("SWTPG_PARTS",)
HIT_MIX = (0, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64)  # unit counts around every slice edge of stride 64


def gpu(test):
    skip = pytest.mark.skipif(any(v in os.environ for v in TUNING_AIDS), reason="a tuning aid is set: launches leave the default geometry")
    return pytest.mark.gpu(skip(test))


def sms() -> int:
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def ragged_units(seed: int, n_links: int, stride: int, specials=()):
    """Seeded per-link unit counts in [0, stride], with each of `specials` on a few links spread over the whole range."""
    rng = np.random.default_rng(seed)
    nu = rng.integers(0, stride + 1, n_links).astype(np.uint32)
    specials = [s for s in specials if s <= stride]
    at = rng.choice(n_links, size=min(n_links, 4 * len(specials)), replace=False)
    for i, l in enumerate(at):
        nu[l] = specials[i % len(specials)]
    return nu


def host_batches(fmt, seed, rate, n_links, stride, nus, gen_kw=None):
    """[(units [links][stride][unit bytes], n_units)]: batch k holds units [k stride, (k + 1) stride) of every link."""
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    p = S.gen_params(seed, rate, **(gen_kw or {}))
    return [(gen(p, n_links, stride, unit0=k * stride), nu) for k, nu in enumerate(nus)]


def run_device(fmt, n_links, stride, nus, params, *, link_kw=None, thresholds=None, rs_factors=None, tp_capacity=1 << 24, **handle):
    """Launches of one handle on frames generated on the device: launch k reads units [k stride, (k + 1) stride) of every link,
    nus[k] of them per link (None: all). Before start, links are configured by link_kw {link: set_link_config kwargs}, their
    thresholds by thresholds {link: table} and the RS memory factors by rs_factors [links][channels]. Asserts that every unit
    was processed once. Returns (TP list of each launch, per-link state, counters [+ "sort": sort stats])."""
    import torch

    gen = S.gen_wib2_device if fmt == "wib2" else S.gen_wibeth_device
    buf = torch.empty(n_links * stride * unit_bytes(fmt), dtype=torch.uint8, device="cuda")
    got = []
    try:
        with S.TPGenerator(n_links, stride, fmt=fmt, tp_capacity=tp_capacity, **handle) as g:
            for l, kw in (link_kw or {}).items():
                g.set_link_config(l, **kw)
            for l, t in (thresholds or {}).items():
                g.set_link_thresholds(l, t)
            if rs_factors is not None:
                g.set_rs_memory_factor(rs_factors)
            g.start()
            for k, nu in enumerate(nus):
                gen(params, buf.data_ptr(), n_links, stride, unit0=k * stride)
                torch.cuda.synchronize()  # the generator runs on the legacy stream, the handle on its own
                g.process_device(buf.data_ptr(), stride, n_units=nu)
                got.append(g.fetch_tps(cap=tp_capacity))  # waits for the launch: the buffer is free to be rewritten
            states = dump_states(g)
            info = g.counters()
            if handle.get("sorted_tps"):
                info["sort"] = g.sort_stats()
    finally:
        del buf
        torch.cuda.empty_cache()
    units = sum(n_links * stride if nu is None else int(nu.sum()) for nu in nus)
    assert info["units_processed"] == units, f"{info['units_processed']} units processed, {units} given"
    return got, states, info


def replay_links(n_links, oracle_of, units_of, cap=1 << 20):
    """Link l's unit arrays units_of(l) (an iterable, in order) through oracle_of(l), one link per worker of a thread pool (ctypes
    releases the GIL). Returns (TPs of each link, per-link state)."""
    def one(l):
        o = oracle_of(l)
        parts = [np.zeros(0, dtype=F.TP_DTYPE)] + [o.process(u, cap=cap) for u in units_of(l) if len(u)]
        return np.concatenate(parts), o.state()

    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        res = list(ex.map(one, range(n_links)))
    return [r[0] for r in res], np.stack([r[1] for r in res])


def replay_oracles(fmt, n_links, stride, nus, params, oracle_of, cap=1 << 18):
    """run_device's launches on the CPU. The generator is counter-based, so each link's units are generated on the host, in
    replay_links's worker of that link, and run through that link's oracle_of(link). Returns (TPs of each link, per-link
    state)."""
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host

    def units_of(l):
        for k, nu in enumerate(nus):
            n = stride if nu is None else int(nu[l])
            if n:
                yield gen(params, 1, n, link0=l, unit0=k * stride, n_threads=1)[0]

    return replay_links(n_links, oracle_of, units_of, cap)


def run_host(fmt, handle, batches, *, link_kw=None, thresholds=None, rs_tables=None):
    """host_batches through one handle (process_host). Links are configured by link_kw {link: set_link_config kwargs} and
    thresholds {link: table} before start, and by rs_tables {link: per-channel RS memory factors} after it, as a frame
    processor sets them. Returns (TPs of all batches, per-link state)."""
    n_links, stride = batches[0][0].shape[:2]
    with S.TPGenerator(n_links, stride, fmt=fmt, **handle) as g:
        for l, kw in (link_kw or {}).items():
            g.set_link_config(l, **kw)
        for l, t in (thresholds or {}).items():
            g.set_link_thresholds(l, t)
        g.start()
        for l, t in (rs_tables or {}).items():
            g.set_link_rs_memory_factor(l, t)
        got = np.concatenate([g.process_host(u, n_units=nu, cap=1 << 22) for u, nu in batches])
        return got, dump_states(g)


def replay_batches(batches, oracle_of):
    """host_batches on the CPU, link l through oracle_of(l): (TPs of all batches, per-link state)."""
    def units_of(l):
        return [u[l, : (u.shape[1] if nu is None else int(nu[l]))] for u, nu in batches]

    tps, state = replay_links(batches[0][0].shape[0], oracle_of, units_of)
    return np.concatenate(tps), state


def assert_links_match(what, fmt, handle, link_kw, got, gstate, want, ostate, min_tps=1):
    assert got.size >= min_tps, f"{what}: only {got.size} TPs"
    assert_same_tps(got, want, what)
    assert_same_state(gstate, ostate, fmt, lambda l: full_conf(handle, link_kw.get(l, {}))["algorithm"], what)


def check(what, fmt, handle, batches, *, link_kw=None, thresholds=None, rs_tables=None, oracle_of=None, min_tps=1):
    """run_host against replay_batches: TPs and carried state of every link. oracle_of defaults to each link's own
    configuration and RS table."""
    link_kw = link_kw or {}
    got, gstate = run_host(fmt, handle, batches, link_kw=link_kw, thresholds=thresholds, rs_tables=rs_tables)
    want, ostate = replay_batches(batches, oracle_of or configured_oracles(fmt, handle, link_kw, rs_tables))
    assert_links_match(what, fmt, handle, link_kw, got, gstate, want, ostate, min_tps)


# ---- the launch rules, restated ---------------------------------------------------------------------------------------------
# swtpg_capi.cu: launch, launch_wibeth, launch_wibeth_geo, and the policies' constants kWarpsPerSm / kFullLoadWarpsPerSm /
# kFullLoadExtraLinks / kQuadCtasPerSm (swtpg_kernels.cuh: PackedSimpleT, PackedRsWibEth, ScalarAlgo, PackedFirIqr,
# PackedFirIqrAnyTaps).
# tests/test_gpu_launch_geometry.py::test_restated_launch_rules_match_the_policy_constants pins the source lines this depends on, so the
# restatement has to be updated together with the rules.
FULL_WARPS_PER_SM = 20   # kFullLoadWarpsPerSm of PackedSimpleT and (inherited) PackedRsWibEth
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
    """[u0, u1) of each slice of a link with n units (wibeth_kernel's slice_of; tests/test_slice_arithmetic.py pins it)."""
    out = []
    for part in range(slices):
        u0 = n - ((n + (1 << part) - 1) >> part)
        u1 = n if part + 1 == slices else n - ((n + (2 << part) - 1) >> (part + 1))
        out.append((u0, u1))
    return out


# ---- host shim ------------------------------------------------------------------------------------------------------------
def linear_map(crate, slot, stream, chan):
    return ((crate * 8 + slot) * 64 + stream) * 64 + chan


def expected_host_tps(tps, link_stream, *, mask=(), tp_timeout=10 ** 9, correct=False, crate=1, slot=0, wib2=False):
    """What process_swtpg_hits makes of device/oracle TP records of one link."""
    out = []
    for r in tps:
        c = int(r["channel"])
        if wib2 or correct:
            off = linear_map(crate, slot, link_stream, c)
        else:  # H2: position-ordered LUT indexed by the frame channel
            off = linear_map(crate, slot, link_stream, int(F.position_to_channel(c)))
        if off in mask:
            continue
        if int(r["time_over_threshold"]) > tp_timeout:
            continue
        out.append((int(r["time_start"]), int(r["time_peak"]), int(r["time_over_threshold"]), off, int(r["adc_integral"]), int(r["adc_peak"])))
    return sorted(out)


def as_tuples(h):
    return sorted((int(r["time_start"]), int(r["time_peak"]), int(r["time_over_threshold"]), int(r["channel"]), int(r["adc_integral"]),
                   int(r["adc_peak"])) for r in h)

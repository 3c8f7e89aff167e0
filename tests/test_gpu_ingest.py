"""The ingest paths at production size, every link against the oracle: the streaming engine (per-link rings, the staging ring,
the gather kernel's ring of bulk copies, registered latency buffers), the frame processors' feeder threads, the pageable bounce
pipeline of swtpg_process_host, and what a TP-buffer overflow delivers.

The sizes are chosen so that each path's bookkeeping turns over: a gather CTA copies far more units than its ring holds, a
link's ring of pending units is reused, a bounce worker reuses each of its two pinned buffers more than once. They are derived
from the library's constants, restated below; test_restated_ingest_constants_match_the_source pins them to the source, so a
changed constant fails there instead of moving a size to the wrong side of its bound."""
import ctypes as C
import os
import re
import threading
from collections import Counter
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import frames as F
from fdreadoutlibs_b200 import hostshim as H
from util import (FIELDS, adc_of, all_wibeth_policies, as_tuples, assert_links_match, assert_same_state, assert_same_tps, check,
                  configured_oracles, dump_states, full_conf, gpu, ragged_units, replay_batches, replay_links, run_host, stats_of,
                  unit_bytes)

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fdreadoutlibs_b200", "csrc")

# ---- the ingest constants, restated ---------------------------------------------------------------------------------------------
# swtpg_stream.cu: gather_units_tma runs kGatherCtas CTAs, each with a ring of kGatherStages stages, kGatherStages - 1 of them in
# flight. A CTA refills a stage (and flips an mbarrier parity) only once it has more than that many units.
GATHER_STAGES = 8
GATHER_CTAS = 64
GATHER_RING_UNITS = (GATHER_STAGES - 1) * GATHER_CTAS  # units per batch above which every gather ring turns over
# swtpg_capi.cu: a pageable source of at least BOUNCE_MIN_BYTES is cut into BOUNCE_CHUNK chunks, dealt round-robin to
# min(BOUNCE_MAX_WORKERS, max(2, cores) / 2) workers with two pinned buffers each.
BOUNCE_CHUNK = 4 << 20
BOUNCE_MIN_BYTES = 16 << 20
BOUNCE_MAX_WORKERS = 8


def bounce_chunks(nbytes: int) -> int:
    return -(-nbytes // BOUNCE_CHUNK)


WAIT_US = 5_000_000  # the longest a submit may wait for ring space before the test fails
# Python feeders submit far slower than a readout's threads, so the engine's default 5 ms dispatch time-out would cut small
# batches; with this one a batch goes out when a link has a full superchunk, as it does at the detector's rate.
DISPATCH_TIMEOUT_US = 200_000


def test_restated_ingest_constants_match_the_source():
    with open(os.path.join(CSRC, "swtpg_stream.cu")) as f:
        stream = f.read()
    with open(os.path.join(CSRC, "swtpg_capi.cu")) as f:
        capi = f.read()

    def one(src, pattern):
        m = re.findall(pattern, src)
        assert len(m) == 1, f"{pattern!r}: {len(m)} matches"
        return m[0]

    assert int(one(stream, r"constexpr int kGatherStages = (\d+);")) == GATHER_STAGES
    assert int(one(stream, r"constexpr unsigned kGatherCtas = (\d+);")) == GATHER_CTAS
    one(stream, r"std::min<unsigned>\(kGatherCtas, b\.n_items\)")                  # one CTA per unit below kGatherCtas units
    one(stream, r"gather_units_tma<kGatherStages><<<")
    one(stream, r"for \(uint32_t k = 0; k < mine && k < STAGES - 1; \+\+k\)\s*load\(k\);")  # STAGES - 1 units in flight
    one(stream, r"if \(k \+ STAGES - 1 < mine\)\s*load\(k \+ STAGES - 1\);")        # the refill
    assert int(one(capi, r"constexpr size_t kBounceChunk = size_t\((\d+)\) << 20;")) << 20 == BOUNCE_CHUNK
    assert int(one(capi, r"constexpr size_t kBounceMinBytes = size_t\((\d+)\) << 20;")) << 20 == BOUNCE_MIN_BYTES
    one(capi, r"const unsigned hw = std::max\(2u, std::thread::hardware_concurrency\(\)\);")
    assert int(one(capi, r"const unsigned workers = std::min\((\d+)u, hw / 2\);")) == BOUNCE_MAX_WORKERS
    one(capi, r"for \(size_t c = t; c < n_chunks && e == cudaSuccess; c \+= workers, \+\+used\)")  # round-robin over workers
    one(capi, r"if \(used >= 2\)\s*e = cudaEventSynchronize\(w\.free_ev\[slot\]\);")              # two buffers per worker
    one(capi, r"if \(bytes >= kBounceMinBytes && is_pageable\(frames\)\)")


# ---- streaming harness ----------------------------------------------------------------------------------------------------------
def feed(g, counts, src_of, *, n_feeders=4, burst=16, late=None, lag=None, lag_units=80, poll_cap=4096):
    """Submits units [0, counts[l]) of every link l, payload src_of(l, u), from n_feeders Python threads that each serve a block
    of links, `burst` units per link and turn, while a poller thread takes TPs `poll_cap` records at a time. Link `late` (its
    own thread) delivers nothing until every other link has passed its third superchunk; link `lag` stays `lag_units` behind
    its feeder's turns. Returns every TP after drain()."""
    n_links, M = len(counts), g.max_units
    submitted = np.zeros(n_links, dtype=np.int64)
    others_past = threading.Event()
    stop = threading.Event()
    errors, parts = [], []
    normal = [l for l in range(n_links) if l != late]

    def submit_upto(l, n):
        while submitted[l] < n:
            u = int(submitted[l])
            if not g.submit(l, src_of(l, u), wait_us=WAIT_US):
                raise AssertionError(f"link {l} unit {u}: no ring space for {WAIT_US} us")
            submitted[l] = u + 1

    def feeder(links):
        try:
            r = 0
            while any(submitted[l] < counts[l] for l in links) and not errors:
                for l in links:
                    want = burst * (r + 1) - (lag_units if l == lag else 0)
                    submit_upto(l, min(int(counts[l]), max(0, want)))
                if not others_past.is_set() and all(submitted[l] > 3 * M for l in normal):
                    others_past.set()
                r += 1
        except Exception as e:  # reported by the test's thread
            errors.append(e)

    def late_feeder():
        try:
            assert others_past.wait(120), "the other links never passed their third superchunk"
            submit_upto(late, int(counts[late]))
        except Exception as e:
            errors.append(e)

    def poller():
        try:
            while not stop.is_set():
                parts.append(g.poll(cap=poll_cap, wait_us=10_000))
        except Exception as e:
            errors.append(e)

    blocks = np.array_split(np.array(normal), n_feeders)
    threads = [threading.Thread(target=feeder, args=([int(l) for l in b],)) for b in blocks]
    if late is not None:
        threads.append(threading.Thread(target=late_feeder))
    pt = threading.Thread(target=poller)
    pt.start()
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    stop.set()
    pt.join()
    if errors:
        raise errors[0]
    assert (submitted == counts).all()
    parts.append(g.drain())
    return np.concatenate(parts)


def check_stream(what, g, fmt, counts, tps, want, ostate, algorithm_of, zero_copy):
    """TPs and state of every link against the oracle, and the counters: every unit once, zero_copy of them by address, the
    gather rings turned over, the timing counts every batch."""
    total = int(np.sum(counts))
    assert tps.size > 1000, f"{what}: only {tps.size} TPs"
    assert_same_tps(tps, np.concatenate(want), what)
    assert_same_state(dump_states(g), ostate, fmt, algorithm_of, what)
    c = g.counters()
    assert c["units_processed"] == total and c["h2d_bytes"] == total * unit_bytes(fmt), c
    assert (c["units_zero_copy"], c["units_staged"]) == (zero_copy, total - zero_copy), c
    assert c["tps_emitted"] == tps.size and c["tps_dropped_overflow"] == 0, c
    assert c["units_processed"] / c["batches"] > GATHER_RING_UNITS, f"{what}: {c['batches']} batches of {total} units"
    assert g.stream_timing()[2] == c["batches"]


def ragged_counts(n_links, n_units):
    return np.array([n_units - 7 * (l % 5) for l in range(n_links)], dtype=np.int64)


# ---- A. the streaming engine at the production geometry ----------------------------------------------------------------------------
PROD_LINKS, PROD_UNITS, PROD_M = 240, 320, 64
LATE, LAG, WRAP = PROD_LINKS - 1, 120, 2
_prod_oracle = {}


def production_units():
    return S.gen_wibeth_host(S.gen_params(700, 0.05), PROD_LINKS, PROD_UNITS)


def production_link_kw():
    policies = all_wibeth_policies()
    return {l: policies[l % len(policies)] for l in range(PROD_LINKS)}


def production_oracle(units, counts):
    """(TPs of each link, state) of the oracle over every link's units: the same for every payload source."""
    if not _prod_oracle:
        _prod_oracle["r"] = replay_links(PROD_LINKS, configured_oracles("wibeth", {}, production_link_kw()),
                                         lambda l: [units[l, : counts[l]]])
    return _prod_oracle["r"]


@gpu
@pytest.mark.parametrize("source", ["registered", "staged", "mixed"])
def test_streaming_production_geometry(source):
    """240 links, superchunks of 64 frames, 4 batch slots, about 320 frames per link (ragged): every link's pending ring and
    the staging ring are reused, every gather CTA copies some 200 units per batch. The six WIBEth policies round-robin over the
    links; four feeder threads in bursts, a late link, a lagging link, a poller that takes 4096 records at a time.
    registered: one latency buffer; staged: unregistered memory, with ADC statistics on; mixed: even links from the latency
    buffer, odd links from temporaries, link 2 from a registered ring whose wrap falls inside a superchunk."""
    units = production_units()
    counts = ragged_counts(PROD_LINKS, PROD_UNITS)
    link_kw = production_link_kw()
    ring, shift = None, 37
    if source == "mixed":  # unit u of link WRAP at slot (u + shift) % n: the wrap lies inside its fifth superchunk
        n = int(counts[WRAP])
        assert (n - shift) % PROD_M != 0 and 4 * PROD_M < n - shift < 5 * PROD_M
        ring = np.ascontiguousarray(np.roll(units[WRAP, :n], shift, axis=0))

    def src_of(l, u):
        if source == "mixed":
            if l == WRAP:
                return ring[(u + shift) % len(ring)]
            return units[l, u] if l % 2 == 0 else units[l, u].copy()
        return units[l, u]

    with S.TPGenerator(PROD_LINKS, PROD_M, adc_stats=source == "staged", dispatch_timeout_us=DISPATCH_TIMEOUT_US) as g:
        assert g.cfg.n_slots == 0  # the default: 4 slots
        for l, kw in link_kw.items():
            g.set_link_config(l, **kw)
        if source == "registered":
            g.register_buffer(units.reshape(-1))
        elif source == "mixed":
            g.register_buffer(units.reshape(-1))
            g.register_buffer(ring.reshape(-1))
        g.start()
        tps = feed(g, counts, src_of, late=LATE, lag=LAG)
        want, ostate = production_oracle(units, counts)
        total = int(counts.sum())
        zero_copy = {"registered": total, "staged": 0, "mixed": int(counts[0::2].sum())}[source]
        check_stream(f"streaming, {source}", g, "wibeth", counts, tps, want, ostate, lambda l: full_conf({}, link_kw[l])["algorithm"],
                     zero_copy)
        if source == "staged":  # batch slots were recycled under load: the statistics kernel read each batch before its reuse
            got = g.read_adc_stats()
            with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
                stats = np.stack(list(ex.map(lambda l: stats_of(adc_of("wibeth", units[l, : counts[l]])), range(PROD_LINKS))))
            for f in ("samples", "sum", "sum_sq", "min", "max"):
                bad = np.argwhere(got[f] != stats[f])
                assert bad.size == 0, f"ADC statistics: {len(bad)} (link, channel) differ in {f}, first {tuple(bad[0])}"
        g.stop()
    del ring, units


# ---- B. WIB2 through the streaming engine ----------------------------------------------------------------------------------------
WIB2_POLICIES = [dict(algorithm="SimpleThreshold", threshold=30), dict(algorithm="FIR", threshold=5), dict(algorithm="AbsRS", threshold=20)]


@gpu
def test_streaming_wib2_at_size():
    """60 links of WIB2 superchunks (5664 B), about 320 each, 64 per batch: each gather CTA copies some 60 units per batch.
    SimpleThreshold, FIR + IQR and AbsRS round-robin; even links from a registered buffer, odd links staged."""
    n_links, n_units, M = 60, 320, 64
    units = S.gen_wib2_host(S.gen_params(710, 0.05), n_links, n_units)
    counts = ragged_counts(n_links, n_units)
    link_kw = {l: WIB2_POLICIES[l % 3] for l in range(n_links)}
    with S.TPGenerator(n_links, M, fmt="wib2", dispatch_timeout_us=DISPATCH_TIMEOUT_US) as g:
        for l, kw in link_kw.items():
            g.set_link_config(l, **kw)
        g.register_buffer(units.reshape(-1))
        g.start()
        tps = feed(g, counts, lambda l, u: units[l, u] if l % 2 == 0 else units[l, u].copy(), late=n_links - 1, lag=17)
        want, ostate = replay_links(n_links, configured_oracles("wib2", {}, link_kw), lambda l: [units[l, : counts[l]]])
        check_stream("WIB2 streaming", g, "wib2", counts, tps, want, ostate, lambda l: full_conf({}, link_kw[l])["algorithm"],
                     int(counts[0::2].sum()))
        g.stop()
    del units


# ---- C. registered ranges changing during a run --------------------------------------------------------------------------------------
def aligned(nbytes, align):
    """A uint8 array of nbytes whose address is a multiple of align, and the allocation that holds it."""
    base = np.zeros(nbytes + align, dtype=np.uint8)
    off = (-base.ctypes.data) % align
    return base[off: off + nbytes], base


@gpu
def test_registered_ranges_during_a_run():
    """One run of 6 WIBEth links (superchunks of 8 frames, 48 frames each), polled after every round of submits:
    link 0: units 8 bytes into a registered array (not 16-byte aligned): staged.
    link 1: a registered range that ends in the middle of unit 24: units 0-23 by address, the rest staged.
    link 2: two page-aligned ranges, adjacent in memory and registered one by one; its units run from the first into the
            second, unit 20 across the seam (staged): the link's range cache misses and reloads.
    links 3, 4: units 0-23 from latency buffer L1; after the third superchunk L1 is unregistered and L2 registered, and the
            links continue from L2.
    link 5: all units from L2's memory: staged while L2 is unregistered (a cached gap), by address once it is registered.
    The split between by-address and staged units is restated per unit from the registered ranges and must be exact."""
    n, M, n_units, ub = 6, 8, 48, F.WIBETH_FRAME_BYTES
    page = os.sysconf("SC_PAGE_SIZE")
    units = S.gen_wibeth_host(S.gen_params(720, 0.3), n, n_units)
    half = n_units // 2
    whole, _w = aligned((n_units + 1) * ub, page)
    short, _s = aligned(n_units * ub, page)
    size_a = -(-(3600 + half * ub) // page) * page
    size_b = -(-(3600 + (n_units - 21) * ub) // page) * page
    ab, _ab = aligned(size_a + size_b, page)
    start2 = size_a - 20 * ub - 3600  # unit 20 of link 2 straddles the seam
    l1, _l1 = aligned(2 * half * ub, page)
    l2, _l2 = aligned(3 * n_units * ub, page)
    srcs = [[None] * n_units for _ in range(n)]
    for u in range(n_units):
        srcs[0][u] = whole[8 + u * ub: 8 + (u + 1) * ub]
        srcs[1][u] = short[u * ub: (u + 1) * ub]
        srcs[2][u] = ab[start2 + u * ub: start2 + (u + 1) * ub]
        for k, l in enumerate((3, 4)):
            buf, slot = (l1, k * half + u) if u < half else (l2, k * n_units + u)
            srcs[l][u] = buf[slot * ub: (slot + 1) * ub]
        srcs[5][u] = l2[(2 * n_units + u) * ub: (2 * n_units + u + 1) * ub]
    for l in range(n):
        for u in range(n_units):
            srcs[l][u][:] = units[l, u]
    short_reg = short[: half * ub + 3600]
    ranges = []  # (lo, hi) of every registered range

    def register(g, a):
        g.register_buffer(a)
        ranges.append((a.ctypes.data, a.ctypes.data + a.nbytes))

    def by_address(p):
        a = p.ctypes.data
        return a % 16 == 0 and any(lo <= a and a + ub <= hi for lo, hi in ranges)

    got, zero_copy = [], np.zeros(n, dtype=np.int64)
    with S.TPGenerator(n, M) as g:
        for a in (whole, short_reg, ab[:size_a], ab[size_a:], l1):
            register(g, a)
        g.start()
        for u in range(n_units):
            if u == half:
                got.append(g.drain())
                g.unregister_buffer(l1)
                ranges.remove((l1.ctypes.data, l1.ctypes.data + l1.nbytes))
                register(g, l2)
            for l in range(n):
                zero_copy[l] += by_address(srcs[l][u])
                assert g.submit(l, srcs[l][u], wait_us=WAIT_US)
            got.append(g.poll())
        got.append(g.drain())
        c = g.counters()
        state = dump_states(g)
        g.stop()
    assert zero_copy.tolist() == [0, half, n_units - 1, n_units, n_units, half]
    assert (c["units_zero_copy"], c["units_staged"]) == (int(zero_copy.sum()), n * n_units - int(zero_copy.sum())), c
    assert c["units_processed"] == n * n_units and c["h2d_bytes"] == n * n_units * ub, c
    want, ostate = replay_links(n, configured_oracles("wibeth", {}), lambda l: [units[l]])
    assert_links_match("registered ranges", "wibeth", {}, {}, np.concatenate(got), state, np.concatenate(want), ostate, min_tps=100)
    assert c["tps_emitted"] == sum(w.size for w in want)


# ---- D. the frame processors driven by feeder threads ----------------------------------------------------------------------------
def check_processors(what, fp, n_links, seqs, oracle_of):
    """Every link's TriggerPrimitives against the oracle over seqs(l), channels through the link's channel map."""
    want, _ = replay_links(n_links, oracle_of, seqs)
    total = 0
    for l in range(n_links):
        got = fp.take_tps(l, cap=1 << 21)
        lut = fp.register_channel_map(l)
        w = sorted((int(r["time_start"]), int(r["time_peak"]), int(r["time_over_threshold"]), int(lut[r["channel"]]), int(r["adc_integral"]),
                    int(r["adc_peak"])) for r in want[l])
        assert as_tuples(got) == w, f"{what}: link {l}: {got.size} TriggerPrimitives, the oracle {len(w)}"
        info = fp.get_info(l)
        assert info["num_frames_dropped_busy"] == 0 and info["num_tps_sent"] == got.size, f"{what}: link {l}: {info}"
        total += got.size
    assert total > 1000


@gpu
@pytest.mark.parametrize("zero_copy", [True, False], ids=["zero_copy", "copy_on_submit"])
def test_frame_processors_with_feeders(zero_copy):
    """FrameProcessors(240, 64) driven as the benchmark drives them: 4 feeder threads in bursts of 16, the buffer played twice.
    Zero-copy from the registered buffer with SimpleThreshold on every link; copy-on-submit with SimpleThreshold and AbsRS
    alternating by link. Every link against the oracle."""
    n_links, n_units, thr = 240, 160, 30
    buf = S.gen_wibeth_host(S.gen_params(730, 0.05), n_links, n_units)
    mixed = not zero_copy
    confs = [dict(algorithm="AbsRS" if mixed and l % 2 else "SimpleThreshold", threshold=thr) for l in range(n_links)]
    link_kw = {l: dict(c, rs_memory_factor=8, rs_scale_factor=5) for l, c in enumerate(confs)}  # conf(): 10 * 0.8, 10 / 2
    with H.FrameProcessors(n_links, 64, threshold=thr, emulator_mode=False, block_on_backpressure=True, n_slots=4,
                           link_confs=confs if mixed else None) as fp:
        if zero_copy:
            fp.register_buffer(buf)
        fp.start()
        st = fp.push_feeders(buf, n_threads=4, burst=16, passes=2)
        fp.stop()
        assert st["payloads"] == 2 * n_links * n_units
        c = fp.counters()
        assert c["units_processed"] == 2 * n_links * n_units, c
        assert (c["units_zero_copy"], c["units_staged"]) == ((c["units_processed"], 0) if zero_copy else (0, c["units_processed"])), c
        assert c["units_processed"] / c["batches"] > GATHER_RING_UNITS, c
        check_processors("feeders", fp, n_links, lambda l: [buf[l], buf[l]], configured_oracles("wibeth", {}, link_kw))
        if zero_copy:
            fp.register_buffer(buf, on=False)


@gpu
def test_frame_processors_paced():
    """40 links fed against the clock at four times real time, blocking on back-pressure."""
    n_links, n_units, thr = 40, 160, 30
    buf = S.gen_wibeth_host(S.gen_params(740, 0.05), n_links, n_units)
    with H.FrameProcessors(n_links, 64, threshold=thr, emulator_mode=False, block_on_backpressure=True) as fp:
        fp.start()
        st = fp.push_feeders(buf, n_threads=4, burst=16, pace=4, passes=2)
        fp.stop()
        assert st["payloads"] == 2 * n_links * n_units
        assert fp.counters()["units_processed"] == 2 * n_links * n_units
        check_processors("paced", fp, n_links, lambda l: [buf[l], buf[l]], configured_oracles("wibeth", dict(threshold=thr)))


# ---- E. the pageable bounce pipeline of swtpg_process_host ---------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n_links,frames", [(1, 2330), (1, 2331), (3, 776), (3, 777)])
def test_bounce_threshold(n_links, frames):
    """Pageable batches just under BOUNCE_MIN_BYTES (one plain copy) and just over it (the bounce workers, the last chunk
    partial and ending inside a frame)."""
    nbytes = n_links * frames * F.WIBETH_FRAME_BYTES
    assert (nbytes >= BOUNCE_MIN_BYTES) == (n_links * frames >= 2331)
    assert nbytes % BOUNCE_CHUNK % F.WIBETH_FRAME_BYTES != 0
    units = S.gen_wibeth_host(S.gen_params(750 + frames, 0.1), n_links, frames)
    check(f"{n_links} x {frames} frames", "wibeth", dict(threshold=30), [(units, None)], min_tps=100)


@gpu
def test_bounce_many_chunks_per_worker():
    """300 links x 64 frames (138 240 000 B): 33 chunks, at least 4 per worker even at 8 workers, so every worker waits for each
    of its buffers at least once. Two batches through one handle (the bounce buffers reused, state carried), the second ragged;
    every WIBEth policy. The same bytes from pinned memory through a second handle give bit-identical TPs and state."""
    n_links, stride = 300, 64
    nbytes = n_links * stride * F.WIBETH_FRAME_BYTES
    assert nbytes >= BOUNCE_MIN_BYTES and bounce_chunks(nbytes) >= 4 * BOUNCE_MAX_WORKERS and nbytes % BOUNCE_CHUNK
    policies = all_wibeth_policies()
    link_kw = {l: policies[l % len(policies)] for l in range(n_links)}
    p = S.gen_params(760, 0.05)
    batches = [(S.gen_wibeth_host(p, n_links, stride, unit0=k * stride), nu)
               for k, nu in enumerate([None, ragged_units(760, n_links, stride, (0, 1, stride))])]
    got, gstate = run_host("wibeth", {}, batches, link_kw=link_kw)
    want, ostate = replay_batches(batches, configured_oracles("wibeth", {}, link_kw))
    assert_links_match("bounce pipeline", "wibeth", {}, link_kw, got, gstate, want, ostate, min_tps=10000)
    pinned = S.PinnedBuffer(2 * nbytes)
    views = [(pinned.array[k * nbytes: (k + 1) * nbytes].reshape(u.shape), nu) for k, (u, nu) in enumerate(batches)]
    try:
        for (v, _), (u, _) in zip(views, batches):
            v[:] = u
        pgot, pstate = run_host("wibeth", {}, views, link_kw=link_kw)
    finally:
        views = v = None
        pinned.close()
    assert np.array_equal(F.sort_tps(pgot), F.sort_tps(got)), "pinned and pageable sources differ"
    assert np.array_equal(pstate, gstate), "pinned and pageable sources leave different state"


@gpu
def test_bounce_wib2():
    """40 links x 80 WIB2 superchunks (18 124 800 B): chunk edges inside superchunks."""
    n_links, stride = 40, 80
    nbytes = n_links * stride * F.WIB2_SUPERCHUNK_BYTES
    assert nbytes >= BOUNCE_MIN_BYTES and BOUNCE_CHUNK % F.WIB2_SUPERCHUNK_BYTES
    link_kw = {l: WIB2_POLICIES[l % 3] for l in range(n_links)}
    units = S.gen_wib2_host(S.gen_params(770, 0.1), n_links, stride)
    check("WIB2 bounce pipeline", "wib2", {}, [(units, None)], link_kw=link_kw, min_tps=1000)


@gpu
def test_bounce_debug_dumps():
    """process_host_debug from a pageable source over the threshold (8 links x 300 frames): the pedestal and waveform dumps
    equal the oracle's on every sample, so every transferred ADC word is checked."""
    n_links, stride = 8, 300
    assert n_links * stride * F.WIBETH_FRAME_BYTES >= BOUNCE_MIN_BYTES
    units = S.gen_wibeth_host(S.gen_params(780, 0.1), n_links, stride)
    with S.TPGenerator(n_links, stride, threshold=30) as g:
        g.start()
        tps, ped, wav = g.process_host(units, debug=True, cap=1 << 21)
    oracles = [configured_oracles("wibeth", dict(threshold=30))(l) for l in range(n_links)]
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        res = list(ex.map(lambda l: oracles[l].process(units[l], dump=True, cap=1 << 20), range(n_links)))
    assert_same_tps(tps, np.concatenate([r[0] for r in res]), "debug dumps")
    for l, (_, p, w) in enumerate(res):
        assert (ped[l] == p).all(), f"pedestal dump of link {l}"
        assert (wav[l] == w).all(), f"waveform dump of link {l}"


# ---- F. overflow keeps true records ----------------------------------------------------------------------------------------------
DENSE = dict(seed=790, rate=4.0, threshold=5)  # some 11 000 TPs per link and 32 frames


def records(a):
    return Counter(zip(*(a[f].tolist() for f in FIELDS)))


def check_overflow(what, delivered, want, c):
    """tps_emitted is the oracle's count, the dropped ones are exactly the ones not delivered, every delivered record is one of
    the oracle's (a sub-multiset: nothing torn, nothing twice)."""
    assert c["tps_emitted"] == want.size, f"{what}: {c['tps_emitted']} TPs emitted, the oracle has {want.size}"
    assert 0 < delivered.size < want.size, what
    assert c["tps_dropped_overflow"] == c["tps_emitted"] - delivered.size, (what, c, delivered.size)
    extra = records(delivered) - records(want)
    assert not extra, f"{what}: {sum(extra.values())} delivered records are none of the oracle's, e.g. {next(iter(extra))}"


@gpu
@pytest.mark.parametrize("sorted_tps", [False, True])
def test_process_host_overflow(sorted_tps):
    n_links, stride, cap = 16, 32, 4096
    units = S.gen_wibeth_host(S.gen_params(DENSE["seed"], DENSE["rate"]), n_links, stride)
    want, _ = replay_links(n_links, configured_oracles("wibeth", dict(threshold=DENSE["threshold"])), lambda l: [units[l]])
    want = np.concatenate(want)
    out = np.zeros(cap, dtype=F.TP_DTYPE)
    n = C.c_size_t(0)
    with S.TPGenerator(n_links, stride, threshold=DENSE["threshold"], tp_capacity=cap, sorted_tps=sorted_tps) as g:
        g.start()
        st = _lib.lib.swtpg_process_host(g._h, units.ctypes.data, None, stride, out.ctypes.data, cap, C.byref(n))
        c = g.counters()
    assert st == _lib.SWTPG_ERR_OVERFLOW and n.value == want.size
    check_overflow("process_host", out, want, c)
    if sorted_tps:
        assert np.array_equal(F.sort_tps(out), out), "the delivered records are not in (time_start, link, channel) order"


@gpu
def test_poll_overflow_keeps_the_records_it_delivered():
    """Streaming with a TP buffer far smaller than a batch's TPs: every poll that reports the overflow still hands over the
    records it copied (SwtpgError.tps), and those are true records."""
    n_links, n_units, M, cap = 16, 32, 8, 2048
    units = S.gen_wibeth_host(S.gen_params(DENSE["seed"], DENSE["rate"]), n_links, n_units)
    want, _ = replay_links(n_links, configured_oracles("wibeth", dict(threshold=DENSE["threshold"])), lambda l: [units[l]])
    want = np.concatenate(want)
    parts, overflows = [], 0

    def poll(g):
        nonlocal overflows
        try:
            part = g.poll()
        except S.SwtpgError as e:
            if e.status != _lib.SWTPG_ERR_OVERFLOW:
                raise
            part, overflows = e.tps, overflows + 1
        parts.append(part)
        return part.size

    with S.TPGenerator(n_links, M, threshold=DENSE["threshold"], tp_capacity=cap) as g:
        g.start()
        for u in range(n_units):
            for l in range(n_links):
                assert g.submit(l, units[l, u], wait_us=WAIT_US)
            poll(g)
        while True:  # drain(), keeping what overflowing polls deliver
            done = g.flush(busy_ok=True)
            g.sync()
            while poll(g) or g.stream_status()[2]:
                pass
            if done and g.stream_status()[0] == 0:
                break
        c = g.counters()
    assert overflows > 0 and c["batches"] >= n_units // M
    check_overflow("poll", np.concatenate(parts), want, c)

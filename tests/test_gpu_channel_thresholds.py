"""Per-channel hit thresholds (swtpg_set_link_thresholds): a threshold table per link for the algorithms whose threshold is in
ADC counts (WIBEth SimpleThreshold, AbsRS, StandardRS; WIB2 SimpleThreshold).

The reference has one tpg_threshold per frame processor. Channels are independent recurrences, so the expected result of a link
with a table is, channel by channel, the uniform oracle run with that channel's threshold (TableOracle). Every link the GPU ran
is compared with it: TPs and carried state."""
import ctypes as C

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import frames as F
from fdreadoutlibs_b200 import hostshim as H
from util import (HANDLE, HIT_MIX, assert_links_match, assert_same_tps, channels, check, dump_states, expected_geometry, full_conf, gpu,
                  host_batches, linear_map, link_config, oracle_for, ragged_units, replay_batches, replay_oracles, run_device, run_host, sms)

# (format, algorithm, handle keyword arguments) of every algorithm a table applies to
IN_SCOPE = [("wibeth", "SimpleThreshold", {}), ("wibeth", "AbsRS", dict(rs_memory_factor=7, rs_scale_factor=2)),
            ("wibeth", "StandardRS", dict(rs_memory_factor=6)), ("wib2", "SimpleThreshold", {})]
EDGES = (0, 1, 16383, 16384, 32767)  # never exceeded from 16383 (SimpleThreshold) or 6555 (running sums) on


def table(seed, fmt, lo=15, hi=80, edges=EDGES, values=None):
    """Seeded thresholds in [lo, hi) (or drawn from `values`) by frame channel, so the two channels of a lane differ, with `edges`
    on a few channels. Few distinct values keep the oracle of the large cases cheap (TableOracle: one run per value)."""
    rng = np.random.default_rng(seed)
    t = (rng.integers(lo, hi, channels(fmt)) if values is None else rng.choice(values, channels(fmt))).astype(np.uint16)
    t[rng.choice(channels(fmt), size=len(edges), replace=False)] = edges
    return t


# ---- the oracle of a link with a table ---------------------------------------------------------------------------------------------
class TableOracle:
    """One link's oracle with per-channel thresholds. The reference has one tpg_threshold per frame processor, and every channel
    is an independent recurrence (nothing in the ADC-threshold algorithms couples two channels), so channel c of a link run with
    a table is channel c of the reference-pinned uniform oracle run with threshold table[c]: its TPs and its carried state. One
    uniform oracle per distinct threshold of the table; table None = the configuration's threshold on every channel."""

    def __init__(self, fmt, conf, link, table=None):
        self.thr = np.full(channels(fmt), conf["threshold"]) if table is None else np.asarray(table, dtype=np.int64)
        self.runs = {int(t): oracle_for(fmt, {**conf, "threshold": int(t)}, link) for t in np.unique(self.thr)}

    def process(self, units, cap=1 << 18):
        parts = [np.zeros(0, dtype=F.TP_DTYPE)]
        for t, o in self.runs.items():
            tps = o.process(units, cap=cap)
            parts.append(tps[self.thr[tps["channel"]] == t])
        return np.concatenate(parts)

    def state(self):
        out = None
        for t, o in self.runs.items():
            st = o.state()
            out = st.copy() if out is None else out
            out[self.thr == t] = st[self.thr == t]
        return out


def table_oracles(fmt, handle, link_kw, tables):
    """oracle_of(link) for links configured by link_kw, with the thresholds of tables {link: table}."""
    return lambda l: TableOracle(fmt, full_conf(handle, link_kw.get(l, {})), l, tables.get(l))


def test_set_link_thresholds_without_handle():
    t = np.zeros(64, dtype=np.uint16)
    assert _lib.lib.swtpg_set_link_thresholds(None, 0, t.ctypes.data) == _lib.SWTPG_ERR_INVALID_ARG
    assert _lib.lib.swtpg_set_link_thresholds(None, 0, None) == _lib.SWTPG_ERR_INVALID_ARG


# ---- every policy against the oracle ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("fmt,algorithm,kw", IN_SCOPE)
def test_packed_policies_with_tables(fmt, algorithm, kw):
    """The packed policy of each algorithm (PackedSimpleT<true>, PackedRsWibEth<false/true>, PackedSimpleWib2): most links with a
    table of their own (the two channels of a lane differ; entries 0, 1, 16383, 16384 and 32767), every third one without.
    Three ragged batches with empty links, state carried."""
    n, stride = (12, 8) if fmt == "wib2" else (24, 16)
    handle = dict(algorithm=algorithm, threshold=40, **kw)
    tables = {l: table(310 + l, fmt) for l in range(n) if l % 3}
    nus = [ragged_units(310 + k, n, stride, (0, 1, stride)) for k in range(3)]
    check(f"{fmt} {algorithm}", fmt, handle, host_batches(fmt, 310, 0.3, n, stride, nus), thresholds=tables,
          oracle_of=table_oracles(fmt, handle, {}, tables), min_tps=1000)


# acc_limit 0 or 1001 and a WIB2 threshold above 32767 are outside the packed policies' validity ranges: ScalarAlgo runs
SCALAR = [("wibeth", "SimpleThreshold", dict(acc_limit=0)), ("wibeth", "AbsRS", dict(acc_limit=1001, rs_memory_factor=7, rs_scale_factor=2)),
          ("wibeth", "StandardRS", dict(acc_limit=0, rs_memory_factor=6)), ("wib2", "SimpleThreshold", dict(threshold=40000))]


@gpu
@pytest.mark.parametrize("fmt,algorithm,kw", SCALAR)
def test_scalar_fallbacks_with_tables(fmt, algorithm, kw):
    """ScalarAlgo with a table on most links. The WIB2 configuration's threshold 40000 is negative as an int16, so a link
    without a table is over threshold on every sample, as in the reference; with a table its channels run their own."""
    n, stride = (9, 8) if fmt == "wib2" else (24, 16)
    handle = dict(algorithm=algorithm, **{"threshold": 40, **kw})
    tables = {l: table(320 + l, fmt) for l in range(n) if l % 3}
    nus = [ragged_units(320 + k, n, stride, (0, 1, stride)) for k in range(3)]
    check(f"scalar {fmt} {algorithm}", fmt, handle, host_batches(fmt, 320, 0.3, n, stride, nus), thresholds=tables,
          oracle_of=table_oracles(fmt, handle, {}, tables), min_tps=500)


@gpu
@pytest.mark.parametrize("fmt,algorithm,kw", IN_SCOPE)
def test_all_equal_table_is_bit_identical_to_no_table(fmt, algorithm, kw):
    n, stride = (8, 8) if fmt == "wib2" else (16, 16)
    nus = [ragged_units(330 + k, n, stride, (0, 1, stride)) for k in range(2)]
    batches = host_batches(fmt, 330, 0.3, n, stride, nus)
    want_tps, want_state = run_host(fmt, dict(algorithm=algorithm, threshold=35, **kw), batches)
    got_tps, got_state = run_host(fmt, dict(algorithm=algorithm, threshold=70, **kw), batches,
                                  thresholds={l: np.full(channels(fmt), 35, dtype=np.uint16) for l in range(n)})
    assert want_tps.size > 100
    assert_same_tps(got_tps, want_tps, "all-equal tables")
    assert (got_state == want_state).all()


# ---- production geometry ----------------------------------------------------------------------------------------------------------
@gpu
def test_mixed_handle_at_production_geometry():
    """SimpleThreshold, AbsRS and StandardRS groups in one handle, each sized from the SM count into the 20-warps-per-SM sliced
    regime, links of the three interleaved; two thirds of the links have tables (drawn from a few, so that neighbouring links of
    a group differ). Ragged unit counts around every slice edge, then a full launch: state carried across slices and launches."""
    per = 20 * sms() + 1
    for algo in ("SimpleThreshold", "AbsRS", "StandardRS"):
        assert expected_geometry(algo, per, 64, sms()) == (20, 4)
    n = 3 * per
    rng = np.random.default_rng(340)
    kinds = np.array([0] * per + [1] * per + [2] * per)
    rng.shuffle(kinds)
    kinds_kw = [dict(threshold=30), dict(algorithm="AbsRS", threshold=30), dict(algorithm="StandardRS", threshold=30, rs_memory_factor=6)]
    link_kw = {l: kinds_kw[int(k)] for l, k in enumerate(kinds)}
    pool = [table(340 + i, "wibeth", edges=(0, 16384), values=(20, 35, 50, 70)) for i in range(7)]
    tables = {l: pool[int(rng.integers(len(pool)))] for l in range(n) if rng.random() < 2 / 3}
    stride = 64
    nus = [ragged_units(340, n, stride, HIT_MIX), None]
    p = S.gen_params(340, 0.1)
    got, gstate, _ = run_device("wibeth", n, stride, nus, p, link_kw=link_kw, thresholds=tables)
    want, ostate = replay_oracles("wibeth", n, stride, nus, p, table_oracles("wibeth", {}, link_kw, tables))
    assert_links_match("mixed production geometry", "wibeth", {}, link_kw, np.concatenate(got), gstate, np.concatenate(want), ostate,
                       min_tps=100000)


@gpu
def test_wib2_ctas_take_several_links_with_tables():
    """WIB2 SimpleThreshold with 20 x SMs links, so every persistent CTA takes several links; each of a link's four channel
    groups reads its own row of the link's table."""
    n = 20 * sms()
    rng = np.random.default_rng(350)
    pool = [table(350 + i, "wib2", edges=(1, 32767), values=(25, 45, 65)) for i in range(5)]
    tables = {l: pool[int(rng.integers(len(pool)))] for l in range(n) if l % 4}
    nus = [ragged_units(350 + k, n, 16, (0, 1, 16)) for k in range(2)]
    p = S.gen_params(350, 0.3)
    got, gstate, _ = run_device("wib2", n, 16, nus, p, thresholds=tables, threshold=60)
    want, ostate = replay_oracles("wib2", n, 16, nus, p, table_oracles("wib2", dict(threshold=60), {}, tables))
    assert_links_match("WIB2 several links per CTA", "wib2", dict(threshold=60), {}, np.concatenate(got), gstate, np.concatenate(want),
                       ostate, min_tps=10000)


# ---- streaming path -----------------------------------------------------------------------------------------------------------------
@gpu
def test_streaming_path_with_tables():
    n, n_units = 8, 12
    link_kw = {l: [dict(threshold=30), dict(algorithm="AbsRS", threshold=30)][l % 2] for l in range(n)}
    tables = {l: table(360 + l, "wibeth") for l in range(n) if l != 3}
    units = S.gen_wibeth_host(S.gen_params(360, 0.3), n, n_units)
    want, _ = replay_batches([(units, None)], table_oracles("wibeth", {}, link_kw, tables))
    with S.TPGenerator(n, 4, sorted_tps=True) as g:
        for l, kw in link_kw.items():
            g.set_link_config(l, **kw)
        for l, t in tables.items():
            g.set_link_thresholds(l, t)
        g.start()
        for u in range(n_units):
            for l in range(n):
                assert g.submit(l, units[l, u], wait_us=1_000_000)
        got = g.drain()
    assert want.size > 500
    assert_same_tps(got, want, "streaming with tables")


# ---- call rules -----------------------------------------------------------------------------------------------------------------------
def raw_thresholds(g, link, t):
    a = None if t is None else np.ascontiguousarray(t, dtype=np.uint16)
    return _lib.lib.swtpg_set_link_thresholds(g._h, link, None if a is None else a.ctypes.data)


def raw_config(g, link, **kw):
    return _lib.lib.swtpg_set_link_config(g._h, link, C.byref(link_config(**kw)))


@gpu
def test_call_rules():
    n = 4
    t = table(370, "wibeth")
    with S.TPGenerator(n, 4) as g:
        assert raw_thresholds(g, n, t) == _lib.SWTPG_ERR_INVALID_ARG  # link out of range
        assert raw_thresholds(g, n, None) == _lib.SWTPG_ERR_INVALID_ARG
        bad = t.copy()
        bad[17] = 32768
        assert raw_thresholds(g, 0, bad) == _lib.SWTPG_ERR_INVALID_ARG  # above 32767
        assert raw_config(g, 1, algorithm=_lib.ALGO_FIR_IQR, threshold=5) == _lib.SWTPG_OK
        assert raw_thresholds(g, 1, t) == _lib.SWTPG_ERR_UNSUPPORTED  # FIR + IQR: the threshold multiplies a sigma
        assert raw_thresholds(g, 1, None) == _lib.SWTPG_OK            # clearing is always accepted
        assert raw_thresholds(g, 0, t) == _lib.SWTPG_OK
        assert raw_config(g, 0, algorithm=_lib.ALGO_FIR_IQR, threshold=5) == _lib.SWTPG_ERR_UNSUPPORTED  # a link with a table
        assert raw_config(g, 0, algorithm=_lib.ALGO_ABS_RS, threshold=5) == _lib.SWTPG_OK                # ... may change otherwise
        g.start()
        assert raw_thresholds(g, 2, t) == _lib.SWTPG_ERR_STATE
        assert raw_thresholds(g, 0, None) == _lib.SWTPG_ERR_STATE
        g.stop()
        assert raw_thresholds(g, 2, t) == _lib.SWTPG_OK
    with S.TPGenerator(2, 4, algorithm="FIR", threshold=5) as g:
        assert raw_thresholds(g, 0, t) == _lib.SWTPG_ERR_UNSUPPORTED
        assert raw_config(g, 0, algorithm=_lib.ALGO_SIMPLE_THRESHOLD, threshold=30) == _lib.SWTPG_OK
        assert raw_thresholds(g, 0, t) == _lib.SWTPG_OK
        assert _lib.lib.swtpg_set_link_config(g._h, 0, None) == _lib.SWTPG_ERR_UNSUPPORTED  # back to the handle's FIR + IQR
    t2 = table(371, "wib2")
    with S.TPGenerator(2, 4, fmt="wib2") as g:
        assert raw_config(g, 0, algorithm=_lib.ALGO_ABS_RS, threshold=20) == _lib.SWTPG_OK
        assert raw_thresholds(g, 0, t2) == _lib.SWTPG_ERR_UNSUPPORTED  # WIB2 AbsRS: sigma units too
        assert raw_thresholds(g, 1, t2) == _lib.SWTPG_OK
        assert raw_config(g, 1, algorithm=_lib.ALGO_ABS_RS, threshold=20) == _lib.SWTPG_ERR_UNSUPPORTED


@gpu
def test_tables_persist_and_refused_calls_change_nothing():
    """A table survives stop / start and later swtpg_set_link_config calls; refused calls leave tables and configurations as they
    were; NULL returns a link to its configuration's threshold. Each run is checked against the oracle."""
    n = 6
    batches = host_batches("wibeth", 380, 0.3, n, 16, [None])
    t = {l: table(380 + l, "wibeth") for l in range(n)}
    handle = dict(threshold=40)
    with S.TPGenerator(n, 16, **handle) as g:
        for l in (0, 1, 2, 3):
            g.set_link_thresholds(l, t[l])
        g.start()
        run1 = g.process_host(batches[0][0])
        g.stop()
        # refused: a table above 32767 on link 4, link 1 with a table moved to FIR + IQR
        bad = t[4].copy()
        bad[0] = 40000
        assert raw_thresholds(g, 4, bad) == _lib.SWTPG_ERR_INVALID_ARG
        assert raw_config(g, 1, algorithm=_lib.ALGO_FIR_IQR, threshold=5) == _lib.SWTPG_ERR_UNSUPPORTED
        g.set_link_config(0, algorithm="AbsRS", threshold=25)  # the table stays and takes precedence over 25
        g.set_link_thresholds(2, None)                         # back to the configuration's 40
        g.start()
        run2 = g.process_host(batches[0][0])
        state2 = dump_states(g)
    first = {l: t[l] for l in (0, 1, 2, 3)}
    want1, _ = replay_batches(batches, table_oracles("wibeth", handle, {}, first))
    assert_same_tps(run1, want1, "first run")
    link_kw = {0: dict(algorithm="AbsRS", threshold=25)}
    second = {l: t[l] for l in (0, 1, 3)}
    want2, ostate2 = replay_batches(batches, table_oracles("wibeth", handle, link_kw, second))
    assert_links_match("after stop / start", "wibeth", handle, link_kw, run2, state2, want2, ostate2, min_tps=100)


# ---- host shim ----------------------------------------------------------------------------------------------------------------------
def plane(offline):  # the shim's stand-in get_plane_from_offline_channel
    c = offline % 2560
    return 1 if c < 800 else (2 if c < 1568 else 0)


@gpu
@pytest.mark.parametrize("stream", [12, 24])  # offline channels 768..895 (planes 1 and 2), 1536..1663 (planes 2 and 0)
def test_frame_processors_with_plane_thresholds(stream):
    """RawDataProcessorConf::tpg_plane_threshold through FrameProcessors(link_confs=...): each link's TriggerPrimitives equal the
    oracle run with the table its conf() resolves through the channel map (one plane left at tpg_threshold)."""
    n_links, n_units = 2, 16
    crate, slot = 0, 0
    units = S.gen_wibeth_host(S.gen_params(390 + stream, 0.5), n_links, n_units)
    confs = [dict(algorithm="SimpleThreshold", threshold=40, plane_threshold=(20, -1, 60)),
             dict(algorithm="AbsRS", threshold=30, plane_threshold=(15, 45, -1))]
    with H.FrameProcessors(n_links, 8, crate_id=crate, slot_id=slot, first_link_id=stream, emulator_mode=True, correct_channel_lookup=True,
                           link_confs=confs) as fp:
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        got = [fp.take_tps(l) for l in range(n_links)]
    key = lambda a, ch: sorted((int(r["time_over_threshold"]), int(ch(r)), int(r["adc_integral"]), int(r["adc_peak"])) for r in a)
    for l, c in enumerate(confs):
        offline = [linear_map(crate, slot, stream + l, ch) for ch in range(64)]
        planes = {plane(o) for o in offline}
        t = np.array([c["plane_threshold"][plane(o)] if c["plane_threshold"][plane(o)] >= 0 else c["threshold"] for o in offline],
                     dtype=np.uint16)
        assert len(set(t.tolist())) >= 2 or len(planes) == 1
        o = TableOracle("wibeth", {**HANDLE, "rs_memory_factor": 8, **{k: v for k, v in c.items() if k != "plane_threshold"}}, l, t)
        want = o.process(units[l])
        assert want.size > 10
        assert key(got[l], lambda r: r["channel"]) == key(want, lambda r: offline[int(r["channel"])]), f"link {stream + l} ({c})"


def test_wib2_plane_thresholds_need_simple_threshold():
    """CPU: conf() refuses plane thresholds for the WIB2 algorithms whose threshold multiplies an IQR sigma, before any handle."""
    with pytest.raises(H.HostError, match="tpg_plane_threshold"):
        H.FrameProcessors(1, 4, fmt="wib2", link_confs=[dict(algorithm="FIR", threshold=5, plane_threshold=(20, -1, -1))])
    with pytest.raises(H.HostError, match="tpg_plane_threshold"):
        H.FrameProcessors(1, 4, fmt="wib2", link_confs=[dict(algorithm="AbsRS", threshold=20, plane_threshold=(-1, 30, -1))])

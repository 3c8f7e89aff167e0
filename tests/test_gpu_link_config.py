"""Per-link TPG configuration (swtpg_set_link_config): one handle serves links with different algorithms and thresholds.

Every link is compared with the oracle run with THAT link's configuration (one `Oracle` per link, carried across batches):
its TPs and its carried state. The handle groups links whose configurations agree in every field their algorithm reads and
launches the batch kernel once per group, one group after another; a handle whose links share one configuration launches as
it did before links had their own."""
import ctypes as C
import os
import subprocess

import numpy as np

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import hostshim as H
from util import (HANDLE, all_wibeth_policies, as_tuples, assert_links_match, assert_same_tps, check, configured_oracles, dump_states,
                  expected_geometry, expected_host_tps, gpu, halving_slices, host_batches, link_config, oracle_for, ragged_units,
                  replay_batches, replay_oracles, run_device, run_host, sms)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- CPU --------------------------------------------------------------------------------------------------------------------
def test_link_config_layout_matches_the_header(tmp_path):
    """The ctypes mirror of swtpg_link_config has the header's size and field offsets (a C program prints them)."""
    fields = [n for n, _ in _lib.SwtpgLinkConfig._fields_]
    src = tmp_path / "link_config_probe.c"
    src.write_text('#include "swtpg.h"\n#include <stddef.h>\n#include <stdio.h>\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(swtpg_link_config));\n'
                   + "".join(f'  printf("%zu\\n", offsetof(swtpg_link_config, {n}));\n' for n in fields)
                   + '  printf("%u\\n", SWTPG_MAX_LINK_CONFIGS);\n  return 0;\n}\n')
    exe = tmp_path / "link_config_probe"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.SwtpgLinkConfig) == 36
    assert out[1:-1] == [getattr(_lib.SwtpgLinkConfig, n).offset for n in fields]
    assert out[-1] == _lib.MAX_LINK_CONFIGS


def test_set_link_config_without_handle():
    c = _lib.SwtpgLinkConfig()
    c.struct_size = C.sizeof(c)
    assert _lib.lib.swtpg_set_link_config(None, 0, C.byref(c)) == _lib.SWTPG_ERR_INVALID_ARG
    assert _lib.lib.swtpg_set_link_config(None, 0, None) == _lib.SWTPG_ERR_INVALID_ARG


# ---- per-link configurations against the oracle ---------------------------------------------------------------------------
@gpu
def test_wibeth_simple_thresholds_and_accumulator_limits():
    """Four SimpleThreshold configurations interleaved by link % 4; three ragged batches with empty links, state carried."""
    confs = [dict(threshold=30, acc_limit=10), dict(threshold=45, acc_limit=3), dict(threshold=20, acc_limit=25), dict(threshold=60, acc_limit=1)]
    n = 24
    link_kw = {l: confs[l % 4] for l in range(n)}
    nus = [ragged_units(201 + k, n, 16, (0, 1, 16)) for k in range(3)]
    check("simple x4", "wibeth", {}, host_batches("wibeth", 201, 0.3, n, 16, nus), link_kw=link_kw, min_tps=1000)


@gpu
def test_every_wibeth_policy_in_one_handle():
    """SimpleThreshold, AbsRS, StandardRS, FIR (binomial taps), FIR (any taps) and the scalar fallback in one handle, with
    per-link RS memory factors and a per-channel table on one AbsRS link set after start."""
    policies = all_wibeth_policies()
    n = 30
    link_kw = {}
    for l in range(n):
        kw = dict(policies[l % len(policies)])
        if kw["algorithm"] in ("AbsRS", "StandardRS"):
            kw["rs_memory_factor"] = kw["rs_memory_factor"] + l % 3  # per-link factors inside one group
        link_kw[l] = kw
    table = np.random.default_rng(202).integers(0, 13, 64).astype(np.uint16)
    nus = [ragged_units(202 + k, n, 16, (0, 1, 16)) for k in range(3)]
    check("all WIBEth policies", "wibeth", {}, host_batches("wibeth", 202, 0.3, n, 16, nus), link_kw=link_kw, rs_tables={7: table},
          min_tps=1000)


@gpu
def test_wib2_policies_in_one_handle():
    """WIB2 SimpleThreshold, FIR and AbsRS in one handle; one AbsRS threshold is beyond the packed comparator's range, so its
    group runs the exact-threshold tier on every channel group."""
    confs = [dict(algorithm="SimpleThreshold", threshold=60), dict(algorithm="FIR", threshold=5), dict(algorithm="AbsRS", threshold=60),
             dict(algorithm="AbsRS", threshold=22000)]
    n = 12
    link_kw = {l: confs[l % 4] for l in range(n)}
    nus = [ragged_units(203 + k, n, 8, (0, 1, 8)) for k in range(2)]
    check("WIB2 policies", "wib2", {}, host_batches("wib2", 203, 0.3, n, 8, nus), link_kw=link_kw, min_tps=100)


@gpu
def test_production_geometries_per_group():
    """Three groups in one handle, each sized from the SM count into a production regime of its own: SimpleThreshold with
    20 x SMs + 1 links (20 warps per SM, sliced), AbsRS above one round (sliced), FIR + IQR with 4k + 3 links (quads, the
    group's last one partial). Frames generated on the device; two launches, state carried."""
    n_simple, n_rs, n_fir = 20 * sms() + 1, 20 * sms() + 1, 4 * sms() + 3
    assert expected_geometry("SimpleThreshold", n_simple, 64, sms()) == (20, 4)
    assert expected_geometry("AbsRS", n_rs, 64, sms()) == (20, 4)
    assert n_fir % 4 == 3
    assert halving_slices(64, 4) == [(0, 32), (32, 48), (48, 56), (56, 64)]
    n = n_simple + n_rs + n_fir
    kinds = np.array([0] * n_simple + [1] * n_rs + [2] * n_fir)
    np.random.default_rng(204).shuffle(kinds)  # groups interleaved over the link range
    kinds_kw = [dict(threshold=30), dict(algorithm="AbsRS", threshold=30), dict(algorithm="FIR", threshold=5)]
    link_kw = {l: kinds_kw[int(k)] for l, k in enumerate(kinds)}
    stride, nus = 64, [None, None]
    p = S.gen_params(204, 0.1)
    got, gstate, _ = run_device("wibeth", n, stride, nus, p, link_kw=link_kw)
    want, ostate = replay_oracles("wibeth", n, stride, nus, p, configured_oracles("wibeth", {}, link_kw), cap=1 << 16)
    assert_links_match("production geometries", "wibeth", {}, link_kw, np.concatenate(got), gstate, np.concatenate(want), ostate,
                       min_tps=10000)


@gpu
def test_streaming_path_sorted_per_link_configs():
    """Streaming path with SWTPG_FLAG_SORTED_TPS and per-link configurations: every link's records equal the oracle's, and
    each batch's list is in (time_start, link, channel) order."""
    n, n_units = 8, 12
    confs = [dict(threshold=30), dict(threshold=45, acc_limit=4), dict(algorithm="AbsRS", threshold=30), dict(algorithm="FIR", threshold=5)]
    link_kw = {l: confs[l % 4] for l in range(n)}
    units = S.gen_wibeth_host(S.gen_params(205, 0.3), n, n_units)
    want, _ = replay_batches([(units, None)], configured_oracles("wibeth", {}, link_kw))
    with S.TPGenerator(n, 4, sorted_tps=True) as g:
        for l, kw in link_kw.items():
            g.set_link_config(l, **kw)
        g.start()
        for u in range(n_units):
            for l in range(n):
                assert g.submit(l, units[l, u], wait_us=1_000_000)
        got = g.drain()
        batches = g.counters()["batches"]
    assert_same_tps(got, want, "streaming")
    order = [(int(a), int(b), int(c)) for a, b, c in zip(got["time_start"], got["link"], got["channel"])]
    runs = 1 + sum(1 for i in range(1, len(order)) if order[i] < order[i - 1])
    assert runs <= batches, f"{runs} ordered runs in {batches} batches"


# ---- equivalences -------------------------------------------------------------------------------------------------------------
@gpu
def test_links_set_to_the_handle_configuration_change_nothing():
    n = 16
    nus = [ragged_units(206 + k, n, 16, (0, 1, 16)) for k in range(2)]
    batches = host_batches("wibeth", 206, 0.3, n, 16, nus)
    handle = dict(threshold=30)
    a_tps, a_state = run_host("wibeth", handle, batches)
    # every field the handle has, and fields SimpleThreshold does not read changed on some links: still one group
    link_kw = {l: (dict(fir_taps=[1, 2, 3], rs_scale_factor=3) if l % 2 else {}) for l in range(n)}
    b_tps, b_state = run_host("wibeth", handle, batches, link_kw=link_kw)
    assert a_tps.size > 100
    assert_same_tps(b_tps, a_tps, "links set to the handle's configuration")
    assert (a_state == b_state).all()


@gpu
def test_every_link_set_to_b_equals_a_handle_created_with_b():
    n = 16
    nus = [ragged_units(207 + k, n, 16, (0, 1, 16)) for k in range(2)]
    batches = host_batches("wibeth", 207, 0.3, n, 16, nus)
    b = dict(algorithm="AbsRS", threshold=25, acc_limit=5, rs_memory_factor=7, rs_scale_factor=2)
    want_tps, want_state = run_host("wibeth", b, batches)
    got_tps, got_state = run_host("wibeth", dict(threshold=60), batches, link_kw={l: b for l in range(n)})
    assert want_tps.size > 100
    assert_same_tps(got_tps, want_tps, "all links set to B")
    assert (got_state == want_state).all()


# ---- call rules -----------------------------------------------------------------------------------------------------------------
def raw_set(g, link, c):
    return _lib.lib.swtpg_set_link_config(g._h, link, None if c is None else C.byref(c))


@gpu
def test_call_rules():
    n = 18
    with S.TPGenerator(n, 4) as g:
        assert raw_set(g, n, link_config()) == _lib.SWTPG_ERR_INVALID_ARG  # link out of range
        bad = link_config()
        bad.struct_size = 12
        assert raw_set(g, 0, bad) == _lib.SWTPG_ERR_INVALID_ARG
        assert raw_set(g, 0, link_config(algorithm=9)) == _lib.SWTPG_ERR_UNSUPPORTED
        assert raw_set(g, 0, link_config(tap_exponent=15)) == _lib.SWTPG_ERR_INVALID_ARG
        # 15 thresholds besides the handle's own 60: 16 distinct configurations
        for l in range(15):
            assert raw_set(g, l, link_config(threshold=10 + l)) == _lib.SWTPG_OK
        assert raw_set(g, 15, link_config(threshold=99)) == _lib.SWTPG_ERR_INVALID_ARG  # a 17th
        assert raw_set(g, 15, link_config(threshold=12, rs_memory_factor=3)) == _lib.SWTPG_OK  # equal to link 2's for SimpleThreshold
        assert raw_set(g, 14, link_config(threshold=99)) == _lib.SWTPG_OK  # link 14 was the only one with threshold 24
        assert raw_set(g, 16, link_config(threshold=60, fir_taps=(C.c_int16 * 8)(3))) == _lib.SWTPG_OK  # the handle's own
        g.start()
        assert raw_set(g, 0, link_config()) == _lib.SWTPG_ERR_STATE
        assert raw_set(g, 0, None) == _lib.SWTPG_ERR_STATE
        g.stop()
        assert raw_set(g, 0, None) == _lib.SWTPG_OK
    with S.TPGenerator(2, 4, fmt="wib2") as g:
        assert raw_set(g, 0, link_config(algorithm=_lib.ALGO_STANDARD_RS)) == _lib.SWTPG_ERR_UNSUPPORTED
        assert raw_set(g, 0, link_config(algorithm=_lib.ALGO_ABS_RS, threshold=0)) == _lib.SWTPG_ERR_INVALID_ARG


@gpu
def test_stop_reconfigure_start_and_reset():
    """Stop, give links other configurations (one back to the handle's with NULL) and start again: the new configurations run
    on fresh state."""
    n = 8
    batches = host_batches("wibeth", 208, 0.3, n, 16, [None])
    first = {l: dict(algorithm="AbsRS", threshold=30) for l in range(0, n, 2)}
    second = {1: dict(threshold=25), 3: dict(algorithm="FIR", threshold=5), 5: dict(algorithm="StandardRS", threshold=30)}
    with S.TPGenerator(n, 16, threshold=40) as g:
        for l, kw in first.items():
            g.set_link_config(l, **kw)
        g.start()
        tps1 = g.process_host(batches[0][0])
        g.stop()
        for l in first:
            g.set_link_config(l, reset=True)
        for l, kw in second.items():
            g.set_link_config(l, **kw)
        g.start()
        tps2 = g.process_host(batches[0][0])
        state2 = dump_states(g)
    handle = dict(threshold=40)
    want1, _ = replay_batches(batches, configured_oracles("wibeth", handle, first))
    want2, ostate2 = replay_batches(batches, configured_oracles("wibeth", handle, second))
    assert_same_tps(tps1, want1, "first configuration")
    assert_links_match("after reconfiguration", "wibeth", handle, second, tps2, state2, want2, ostate2, min_tps=100)


# ---- host shim ------------------------------------------------------------------------------------------------------------------
@gpu
def test_frame_processors_with_their_own_configurations():
    """Frame processors of one engine whose conf() differ in algorithm and threshold (which the engine refused before links had
    their own configurations): each link's TriggerPrimitives equal the oracle's for its own conf, channel map and algorithm field."""
    n_links, n_units, sc = 4, 13, 4
    units = S.gen_wibeth_host(S.gen_params(209, 0.5), n_links, n_units)
    confs = [dict(algorithm="SimpleThreshold", threshold=25), dict(algorithm="AbsRS", threshold=30),
             dict(algorithm="SimpleThreshold", threshold=40, acc_limit=4), dict(algorithm="AbsRS", threshold=20, rs_memory_factor=0.6)]
    with H.FrameProcessors(n_links, sc, link_confs=confs) as fp:
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        for l, c in enumerate(confs):
            o = oracle_for("wibeth", {**HANDLE, "rs_memory_factor": round(10 * c.get("rs_memory_factor", 0.8)), "rs_scale_factor": 5,
                                      **{k: v for k, v in c.items() if k != "rs_memory_factor"}}, l)
            want = o.process(units[l])
            got = fp.take_tps(l)
            assert want.size > 10
            assert as_tuples(got) == expected_host_tps(want, l), f"link {l} ({c})"
            assert (got["algorithm"] == {"SimpleThreshold": 2, "AbsRS": 3}[c["algorithm"]]).all()

"""The C++ frame-processor shim (fdreadoutlibs_b200/host/): the reference's plug-in interface — conf / start / stop / get_info,
sequence_check + timestamp_check pre-tasks, find_hits post-task, process_swtpg_hits — with the GPU pipeline behind find_hits.
CPU part: the library loads, exports its harness, refuses unknown algorithms the way the reference does and fails loudly
without a device. GPU part: TriggerPrimitives equal the oracle's TPs pushed through the same LUT / mask / timeout logic."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import hostshim as H
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B
from util import HANDLE, adc_of, as_tuples, expected_host_tps, linear_map, oracle_for


def test_host_library_exports():
    lib = C.CDLL(H.HOST_LIB_PATH)
    for name in H.EXPORTS:
        assert hasattr(lib, name), name
    assert C.sizeof(H.HostInfo) == 152 and C.sizeof(H.HostConf) == 160 and H.HOST_TP_DTYPE.itemsize == 48


def test_unknown_algorithm_is_tpg_algorithm_inexistent():
    """conf() throws TPGAlgorithmInexistent for an unknown tpg_algorithm (src/wibeth/WIBEthFrameProcessor.cpp:195-197) — before any
    device is touched."""
    with pytest.raises(H.HostError, match="TPGAlgorithmInexistent"):
        H.FrameProcessors(1, 4, algorithm="NoSuchAlgo")
    with pytest.raises(H.HostError, match="TPGAlgorithmInexistent"):
        H.FrameProcessors(1, 4, fmt="wib2", algorithm="StandardRS")


@pytest.mark.skipif(S.device_available(), reason="needs a box WITHOUT a GPU")
def test_no_cpu_fallback():
    with pytest.raises(H.HostError, match="CUDA"):
        H.FrameProcessors(1, 4)


def test_tpset_windows_heartbeats_and_tardy_cutoff():
    """TPCTPRequestHandler::send_tp_sets (src/TPCTPRequestHandler.cpp:99-193) restated step by step in Python as the checker:
    window [start, newest - min_latency), payload or heartbeat, start/end from the first/last TP, cut-off published, later TPs
    below the cut-off are tardy. CPU only — this component sits after the GPU path and defines its latency budget."""
    rng = np.random.default_rng(5)
    lat = 5000
    tp_t = np.sort(rng.integers(1_000_000, 1_200_000, 400).astype(np.uint64))
    tp_t = tp_t[(tp_t < 1_060_000) | (tp_t > 1_100_000)]  # a 40k-tick hole -> heartbeats
    tps = np.zeros(tp_t.size, dtype=H.HOST_TP_DTYPE)
    tps["time_start"], tps["channel"], tps["adc_integral"] = tp_t, rng.integers(0, 2560, tp_t.size), rng.integers(1, 9999, tp_t.size)
    h = H.TPSetHandler(source_id=9, min_latency_ticks=lat, run_number=42)
    # model
    buf, cutoff, first, start_win, seq, want, tardy = [], 0, True, 0, 0, [], 0
    # TPs arrive in bursts (what a superchunk-batching producer does), each burst shuffled; one burst arrives late
    n_b = tps.size - 60
    bursts = np.array_split(np.arange(n_b), 25) + [np.array([i]) for i in range(n_b, tps.size)]  # the last 60 arrive one by one
    order = list(range(len(bursts)))
    order[10], order[14] = order[14], order[10]  # out-of-order delivery that is still above the cut-off (= time of the last TP sent)
    order.remove(3)
    order.insert(20, 3)                          # burst 3 shows up after ~17 later bursts: every TP in it is tardy
    for b in order:
        idx = rng.permutation(bursts[b])
        accepted = h.receive(tps[idx])
        ok = 0
        for i in idx:
            if int(tps["time_start"][i]) < cutoff:
                tardy += 1
            else:
                buf.append((int(tps["time_start"][i]), int(tps["channel"][i]), int(tps["adc_integral"][i])))
                ok += 1
        assert accepted == ok
        for _ in range(3):  # a few sender cycles per burst
            produced = h.cycle()
            buf.sort()
            exp = False
            if buf:
                newest, oldest = buf[-1][0], buf[0][0]
                if first:
                    start_win, first = oldest, False
                if newest - start_win > lat:
                    end_win = newest - lat
                    objs = [x for x in buf if start_win <= x[0] < end_win]
                    want.append(dict(seqno=seq, type=1 if objs else 2, start_time=objs[0][0] if objs else start_win,
                                     end_time=objs[-1][0] if objs else end_win, n=len(objs), objs=objs))
                    cutoff = want[-1]["end_time"]
                    seq += 1
                    start_win = end_win
                    exp = True
            assert produced == exp
            assert h.cutoff() == cutoff
    got = h.sets()
    assert len(got) == len(want) and len(want) > 10
    for (hdr, objs), w in zip(got, want):
        assert (hdr["seqno"], hdr["type"], hdr["start_time"], hdr["end_time"], hdr["n_objects"]) == (w["seqno"], w["type"], w["start_time"], w["end_time"], w["n"])
        assert hdr["run_number"] == 42 and hdr["origin"] == 9
        assert [(int(o["time_start"]), int(o["channel"]), int(o["adc_integral"])) for o in objs] == w["objs"]
    info = h.info()
    assert tardy > 0 and info["num_tps_suppressed_tardy"] == tardy
    assert info["num_heartbeats"] == sum(1 for w in want if w["type"] == 2) and info["num_heartbeats"] > 0
    assert info["num_tpsets_sent"] == len(want) and info["num_tps_sent"] == sum(w["n"] for w in want)
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("algorithm,algo_id,correct", [("SimpleThreshold", 0, False), ("SimpleThreshold", 0, True), ("AbsRS", 1, False)])
def test_wibeth_frame_processor_end_to_end(algorithm, algo_id, correct):
    n_links, n_units, sc = 3, 21, 4
    units = S.gen_wibeth_host(S.gen_params(61, 0.5), n_links, n_units)
    mask = (linear_map(1, 0, 1, 5), linear_map(1, 0, 2, 40))
    cfg = B.make_config(algorithm=algo_id, threshold=25, rs_memory_factor=8, rs_scale_factor=5)  # conf(): 10*0.8, 10/2
    want, _ = B.oracle_process_links(cfg, units)
    timeout = 32 * 12
    with H.FrameProcessors(n_links, sc, algorithm=algorithm, threshold=25, rs_memory_factor=0.8, rs_scale_factor=2, channel_mask=mask,
                           tp_timeout=timeout, correct_channel_lookup=correct) as fp:
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        assert fp.last_daq_time(0) == int(units[0, -1, 8:16].view("<u8")[0])
        fp.stop()  # flushes the ragged tail (21 = 5 x 4 + 1)
        total_sent = total_long = 0
        for l in range(n_links):
            got = fp.take_tps(l)
            w = want[want["link"] == l]
            assert as_tuples(got) == expected_host_tps(w, l, mask=mask, tp_timeout=timeout, correct=correct), f"link {l}"
            assert (got["detid"] == 3).all() and (got["type"] == 1).all() and (got["version"] == 1).all()
            assert (got["algorithm"] == {"SimpleThreshold": 2, "AbsRS": 3}[algorithm]).all()
            info = fp.get_info(l)
            assert info["num_tps_sent"] == got.size and info["num_ts_errors"] == 1  # first frame: previous_ts = 0
            assert info["num_seq_id_errors"] == 1 and info["num_frames_dropped_busy"] == 0  # first frame: previous_seq_id = 0, seq 0 != 1
            n_long = sum(1 for r in w if int(r["time_over_threshold"]) > timeout and
                         linear_map(1, 0, l, int(F.position_to_channel(int(r["channel"]))) if not correct else int(r["channel"])) not in mask)
            assert info["num_tps_suppressed_too_long"] == n_long
            assert fp.misconfigurations(l) == 0
            # RegisterToChannelNumber: position p holds frame channel 16(p/16) + perm[p%16]
            assert (fp.register_channel_map(l) == [linear_map(1, 0, l, int(F.position_to_channel(p))) for p in range(64)]).all()
            top = info["top"]
            assert len(top) == 10 and all(top[i][1] >= top[i + 1][1] for i in range(9))
            total_sent += got.size
            total_long += n_long
        assert total_sent > 100 and total_long > 0


@pytest.mark.gpu
def test_wibeth_pre_process_checks_and_emulator_mode():
    """sequence_check / timestamp_check count discontinuities (src/wibeth/WIBEthFrameProcessor.cpp:298-405); a wrong geo id is
    reported once (LinkMisconfiguration, :430-432); emulator mode rewrites geo id and timestamps; a full sink counts
    FailedToSendTP-style drops."""
    units = S.gen_wibeth_host(S.gen_params(62, 0.5), 1, 12)
    with H.FrameProcessors(1, 4, threshold=25, slot_id=3) as fp:  # frames carry slot 0
        fp.start()
        for u in (0, 1, 2, 5, 6, 7):  # gap of 3 frames
            fp.push(0, units[0, u].copy())
        fp.stop()
        info = fp.get_info(0)
        # the very first frame already counts (previous ts / seq id start at 0, as in the reference), then the gap
        assert info["num_ts_errors"] == 2 and info["num_seq_id_errors"] == 2
        assert info["max_seq_id_jump"] == 2 and info["min_seq_id_jump"] == -1
        assert fp.error_count(0, "MISSING_FRAMES") == 2 and fp.error_count(0, "SEQUENCE_ID_JUMP") == 2
        assert fp.misconfigurations(0) == 1
    with H.FrameProcessors(1, 4, threshold=25, slot_id=3, emulator_mode=True, sink_capacity=5) as fp:
        fp.start()
        frames = [units[0, u].copy() for u in range(8)]
        for f in frames:
            fp.push(0, f)
        fp.stop()
        ts = [int(f[8:16].view("<u8")[0]) for f in frames]
        assert ts == [2048 * (i + 1) for i in range(8)]          # perfectly incrementing, from previous_ts = 0
        assert all(((int(f[0:8].view("<u8")[0]) >> 22) & 0xF) == 3 for f in frames)  # slot stamped
        info = fp.get_info(0)
        assert info["num_ts_errors"] == 0 and fp.misconfigurations(0) == 0
        got = fp.take_tps(0)
        assert got.size == 5 and info["num_tps_send_failed"] > 0 and info["num_tps_sent"] == 5
    # default back-pressure policy = the reference's try_send: never block, drop and count
    with H.FrameProcessors(1, 1, threshold=25, block_on_backpressure=False) as fp:
        fp.start()
        for rep in range(200):
            for u in range(12):
                fp.push(0, units[0, u].copy())
        fp.stop()
        info = fp.get_info(0)
        assert info["num_frames_dropped_busy"] >= 0  # may or may not trigger; the call must never block or throw


@pytest.mark.gpu
def test_collection_channels_fall_back_to_simple_threshold():
    """enable_simple_threshold_on_collection: R = 0 on plane-0 channels (src/wibeth/WIBEthFrameProcessor.cpp:441-450)."""
    n_units = 16
    crate, slot, stream = 0, 0, 24  # offline channels 1536..1599 of the stand-in map: the upper half is on the collection plane
    units = S.gen_wibeth_host(S.gen_params(63, 0.5), 1, n_units)
    cfg = B.make_config(algorithm=1, threshold=25, rs_memory_factor=8, rs_scale_factor=5)
    o = B.Oracle(cfg)
    fac = np.array([0 if (linear_map(crate, slot, stream, c) % 2560) >= 1568 else 8 for c in range(64)], dtype=np.uint16)
    assert (fac == 0).any() and (fac == 8).any()
    o.set_memory_factor(fac)
    want = o.process(units[0])
    with H.FrameProcessors(1, 8, algorithm="AbsRS", threshold=25, crate_id=crate, slot_id=slot, first_link_id=stream, emulator_mode=True,
                           collection_simple_threshold=True, correct_channel_lookup=True) as fp:
        fp.start()
        for u in range(n_units):
            fp.push(0, units[0, u].copy())
        fp.stop()
        got = fp.take_tps(0)
    # emulator mode rewrote the timestamps (2048, 4096, ...): compare on fields that do not depend on the absolute time
    key = lambda a, ch: sorted((int(r["time_over_threshold"]), int(ch(r)), int(r["adc_integral"]), int(r["adc_peak"])) for r in a)
    assert key(got, lambda r: r["channel"]) == key(want, lambda r: linear_map(crate, slot, stream, int(r["channel"])))
    assert got.size > 50


@pytest.mark.gpu
@pytest.mark.parametrize("algorithm,algo_id", [("SimpleThreshold", 0), ("FIR", 3), ("AbsRS", 1)])
def test_wib2_frame_processor_end_to_end(algorithm, algo_id):
    n_links, n_units = 2, 40
    thr = {0: 30, 3: 5, 1: 20}[algo_id]
    units = S.gen_wib2_host(S.gen_params(64, 0.5), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(fmt="wib2", algorithm=algo_id, threshold=thr), units)
    with H.FrameProcessors(n_links, 8, fmt="wib2", algorithm=algorithm, threshold=thr) as fp:
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        for l in range(n_links):
            got = fp.take_tps(l)
            assert as_tuples(got) == expected_host_tps(want[want["link"] == l], l, wib2=True), f"link {l}"
            assert (got["algorithm"] == 0).all()  # kUnknown: never assigned in the reference (wib2/WIB2FrameProcessor.hpp:137)
            assert fp.get_info(l)["num_ts_errors"] == 1


def wib2_masked_case(seed, n_links=2, n_units=40, threshold=30):
    """WIB2 units of n_links links, the oracle's records of them, a channel mask holding the two busiest channels of every link
    and a tp_timeout that about a quarter of the records exceed."""
    units = S.gen_wib2_host(S.gen_params(seed, 0.5), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(fmt="wib2", threshold=threshold), units)
    mask = []
    for l in range(n_links):
        ch, n = np.unique(want[want["link"] == l]["channel"], return_counts=True)
        mask += [linear_map(1, 0, l, int(c)) for c in ch[np.argsort(-n, kind="stable")[:2]]]
    return units, want, tuple(mask), int(np.percentile(want["time_over_threshold"], 75))


def push_all(fp, units):
    fp.start()
    for u in range(units.shape[1]):
        for l in range(units.shape[0]):
            fp.push(l, units[l, u].copy())
    fp.stop()


@pytest.mark.gpu
def test_wib2_mask_timeout_and_bounded_sink():
    """WIB2FrameProcessor::process_swtpg_hits (src/wib2/WIB2FrameProcessor.cpp:398-479): a masked channel's records are skipped,
    one over tp_timeout is suppressed, one that tp_out refuses is counted as failed, and num_tps_sent counts every record that
    passed the mask whatever became of it (:469-470). The TriggerPrimitives carry Algorithm::kUnknown."""
    units, want, mask, timeout = wib2_masked_case(68)
    n_links = units.shape[0]
    wants = [want[want["link"] == l] for l in range(n_links)]
    unmasked = [[r for r in w if linear_map(1, 0, l, int(r["channel"])) not in mask] for l, w in enumerate(wants)]
    exp = [expected_host_tps(w, l, mask=mask, tp_timeout=timeout, wib2=True) for l, w in enumerate(wants)]
    cap = min(len(e) for e in exp) // 2
    with H.FrameProcessors(n_links, 8, fmt="wib2", threshold=30, channel_mask=mask, tp_timeout=timeout, sink_capacity=cap) as fp:
        push_all(fp, units)
        for l in range(n_links):
            got, info = fp.take_tps(l), fp.get_info(l)
            n_long = sum(1 for r in unmasked[l] if int(r["time_over_threshold"]) > timeout)
            assert cap > 10 and n_long > 0 and len(unmasked[l]) < wants[l].size
            # which records the sink takes depends on the delivery order: each is one of the expected ones
            assert got.size == cap and not Counter(as_tuples(got)) - Counter(exp[l]), f"link {l}"
            assert (got["algorithm"] == 0).all()
            assert info["num_tps_suppressed_too_long"] == n_long and info["num_tps_send_failed"] == len(exp[l]) - cap
            assert info["num_tps_sent"] == len(unmasked[l]) and info["num_frames_dropped_busy"] == 0


@pytest.mark.gpu
def test_wib2_get_info_top_channels():
    """WIB2FrameProcessor::get_info's top channels: the ten offline channels with the most unmasked records
    since the last call, too-long ones included, most first and ties in ascending channel order. The call resets the counts."""
    units, want, mask, timeout = wib2_masked_case(69)
    with H.FrameProcessors(units.shape[0], 8, fmt="wib2", threshold=30, channel_mask=mask, tp_timeout=timeout) as fp:
        push_all(fp, units)
        for l in range(units.shape[0]):
            offline = [linear_map(1, 0, l, c) for c in range(256)]
            n = Counter(linear_map(1, 0, l, int(r["channel"])) for r in want[want["link"] == l])
            n = Counter({c: k for c, k in n.items() if c not in mask})
            info = fp.get_info(l)
            assert info["top"] == [(c, n[c]) for c in sorted(offline, key=lambda c: (-n[c], c))[:10]], f"link {l}"
            assert info["num_tps_sent"] == sum(n.values()) and info["rate_tp_hits"] > 0
            again = fp.get_info(l)
            assert again["top"] == [(c, 0) for c in sorted(offline)[:10]]
            assert again["num_tps_sent"] == again["num_tps_suppressed_too_long"] == again["num_tps_send_failed"] == 0
            assert again["rate_tp_hits"] == 0


@pytest.mark.gpu
def test_wib2_adc_stats_by_offline_channel():
    """get_adc_stats of each WIB2 processor: 256 entries under the offline channels of the frame channels (the direct map), a
    masked channel too; mean, RMS, minimum and maximum as numpy computes them."""
    n_links, n_units = 2, 16
    units = S.gen_wib2_host(S.gen_params(591, 0.3), n_links, n_units)
    masked = linear_map(1, 0, 0, 9)
    with H.FrameProcessors(n_links, 8, fmt="wib2", channel_mask=(masked,), adc_stats=True) as fp:
        assert fp.adc_stats(0).size == 0  # no frame yet: no channel map
        push_all(fp, units)
        got = [fp.adc_stats(l) for l in range(n_links)]
    assert masked in got[0]["offline_channel"]
    for l in range(n_links):
        a = adc_of("wib2", units[l]).astype(np.float64)
        g = got[l]
        assert g.size == 256 and g["offline_channel"].tolist() == [linear_map(1, 0, l, c) for c in range(256)]
        assert (g["samples"] == a.shape[0]).all()
        np.testing.assert_allclose(g["mean"], a.mean(0), rtol=1e-12)
        np.testing.assert_allclose(g["rms"], a.std(0), rtol=1e-9)
        assert g["min"].tolist() == a.min(0).astype(int).tolist() and g["max"].tolist() == a.max(0).astype(int).tolist()


@pytest.mark.gpu
def test_adc_stats_with_per_link_configurations():
    """adc_stats=True together with link_confs: two WIBEth links of one engine with different algorithms. Each link's
    TriggerPrimitives equal the oracle's for its own configuration, and each link's ADC statistics equal numpy's."""
    n_links, n_units = 2, 16
    units = S.gen_wibeth_host(S.gen_params(592, 0.5), n_links, n_units)
    confs = [dict(algorithm="SimpleThreshold", threshold=25), dict(algorithm="AbsRS", threshold=30)]
    with H.FrameProcessors(n_links, 8, link_confs=confs, adc_stats=True) as fp:
        push_all(fp, units)
        got = [fp.take_tps(l) for l in range(n_links)]
        stats = [fp.adc_stats(l) for l in range(n_links)]
    for l, c in enumerate(confs):
        want = oracle_for("wibeth", {**HANDLE, **c}, l).process(units[l])
        assert want.size > 10 and as_tuples(got[l]) == expected_host_tps(want, l), f"link {l} ({c})"
        assert (got[l]["algorithm"] == {"SimpleThreshold": 2, "AbsRS": 3}[c["algorithm"]]).all()
        a = adc_of("wibeth", units[l]).astype(np.float64)
        g = stats[l]
        assert g["offline_channel"].tolist() == [linear_map(1, 0, l, int(F.position_to_channel(c))) for c in range(64)]
        assert (g["samples"] == a.shape[0]).all()
        np.testing.assert_allclose(g["mean"], a.mean(0), rtol=1e-12)
        np.testing.assert_allclose(g["rms"], a.std(0), rtol=1e-9)
        assert g["min"].tolist() == a.min(0).astype(int).tolist() and g["max"].tolist() == a.max(0).astype(int).tolist()


@pytest.mark.gpu
def test_zero_copy_latency_buffer_through_the_frame_processors():
    """find_hits with the payload array registered as the latency buffer (TpgEngine::register_latency_buffer): no per-frame
    copy on the host, identical TriggerPrimitives."""
    n_links, n_units = 12, 40
    units = S.gen_wibeth_host(S.gen_params(66, 0.4), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=25), units)
    payloads = units.copy()
    with H.FrameProcessors(n_links, 8, threshold=25, block_on_backpressure=True) as fp:
        fp.register_buffer(payloads)
        fp.start()
        fp.push_parallel(payloads)
        fp.stop()
        got = [fp.take_tps(l) for l in range(n_links)]
        fp.register_buffer(payloads, on=False)
    for l in range(n_links):
        assert as_tuples(got[l]) == expected_host_tps(want[want["link"] == l], l, slot=l // 8), f"link {l}"


@pytest.mark.gpu
@pytest.mark.parametrize("block", [True, False])
def test_one_thread_per_link_concurrently(block):
    """The reference's threading model (one post-processing thread per link, src/wibeth/WIBEthFrameProcessor.cpp:231): 24 C++
    threads push their links' frames at the same time through swtpg_submit / swtpg_poll. With blocking back-pressure nothing is
    lost and every link's TPs equal the oracle's; with the reference's drop policy (try_send semantics) the call never blocks
    and whatever was dropped is accounted for."""
    n_links, n_units = 24, 48
    units = S.gen_wibeth_host(S.gen_params(65, 0.4), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=25), units)
    with H.FrameProcessors(n_links, 4, threshold=25, block_on_backpressure=block) as fp:
        fp.start()
        fp.push_parallel(units.copy())
        fp.stop()
        dropped = sum(fp.get_info(l)["num_frames_dropped_busy"] for l in range(n_links)) if not block else 0
        got = [fp.take_tps(l) for l in range(n_links)]
    if block:
        for l in range(n_links):
            assert as_tuples(got[l]) == expected_host_tps(want[want["link"] == l], l, slot=l // 8), f"link {l}"
    else:
        assert dropped >= 0 and sum(g.size for g in got) > 0

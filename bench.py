#!/usr/bin/env python
"""bench.py — SWTPG hot-path throughput on B200 (see DESIGN.md §6).

  python bench.py [--gpus N] [--steps K] [--warmup W]            native arm (CUDA kernels through the C ABI)
  python bench.py ... --dump-outputs DIR                         also write the TP list of the last timed step as DIR/tp_<field>.npy
  python bench.py --impl reference [--steps K] [--warmup W]      the reference's own AVX2 code on the host cores

A "step" = one superchunk batch: every link of this GPU's shard advances by `frames` WIBEth frames through the fused
unpack -> pedestal -> hit-finding kernel, state carried from the previous step. Under torchrun each rank owns one GPU
and an independent block of links (no data-path collective); the line printed by rank 0 carries the whole-job aggregate.

  value      the fused kernel on frames resident in HBM (CUDA events around exactly K launches, max over ranks)
  e2e        the drop-in path as a readout application drives it: a few feeder threads push frames of 240 links (6 APAs: what one
             host link carries) through WIBEthFrameProcessor — sequence_check, timestamp_check, find_hits -> swtpg_submit — out of
             a registered latency buffer; the library gathers them over the host link, runs the kernel and hands the
             TriggerPrimitives back. Host buffers in, TPs out, every copy inside the timed region.
  e2e_batch  the batch entry point (swtpg_process_host, one big pinned buffer): the host link's ceiling for this workload

Every timed kernel is checked right after its timing: the state is reset, one more launch runs on the same frames, and the
TPs of four sampled links are compared tuple for tuple with the CPU oracle (`verified_links`).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import resource
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLES_PER_FRAME = 64 * 64
FRAME_BYTES = 7200
APA_SAMPLES_PER_S = 2560 * 62.5e6 / 32  # 2560 channels x 1.953125 MHz = 5.0e9
STATE_BYTES_PER_CHANNEL = 14           # SimpleThreshold: 7 x 16-bit carried values (DESIGN.md §4)
TP_BYTES = 32
METRIC = "adc_samples_per_sec"
UNIT = "samples/s"
REF_US_PER_FRAME_PER_CORE = 2.26       # the reference's AVX2 processing of one frame on one core of the round-1 bench box (1.81 Gsamples/s/core)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--links", type=int, default=5920, help="WIBEth links per GPU (5920 = 148 APAs: config[2]'s module-scale shard)")
    ap.add_argument("--frames", type=int, default=64, help="frames per link per step (superchunk length)")
    ap.add_argument("--threshold", type=int, default=60)
    ap.add_argument("--pulse-rate", type=float, default=0.02, help="pulses per channel per 64 ticks")
    ap.add_argument("--stream-links", type=int, default=240, help="links of the streaming (plug-in) run per GPU: 240 = 6 APAs")
    ap.add_argument("--stream-units", type=int, default=512, help="frames per link in the streaming run's latency buffer")
    ap.add_argument("--stream-passes", type=int, default=16)
    ap.add_argument("--feeders", type=int, default=4, help="feeder threads of the streaming run per GPU")
    ap.add_argument("--module-links", type=int, default=6000, help="config[2] as written: links of the whole module, split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the FIR / running-sum / WIB2 / stress side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the TP list of the last timed step (rank 0's links) to DIR/tp_<field>.npy")
    return ap.parse_args()


DUMP_MAX_BYTES = 64 << 20


def dump_tps(out_dir: str, tps):
    """One float64 array per TP field, in the canonical (time_start, link, channel) order, so that two builds can be compared
    element for element (every field fits float64 exactly: timestamps stay below 2^53). A list over DUMP_MAX_BYTES is cut
    to a fixed, seeded sample of its rows."""
    import numpy as np

    from fdreadoutlibs_b200 import frames as F

    tps = F.sort_tps(tps)
    names = tps.dtype.names
    keep = DUMP_MAX_BYTES // (8 * len(names))
    if tps.size > keep:
        tps = tps[np.sort(np.random.default_rng(0).choice(tps.size, keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name in names:
        np.save(os.path.join(out_dir, f"tp_{name}.npy"), tps[name].astype(np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons, sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period_ms: int = 200):
        self.rows, self.proc, self.index, self.period_ms = [], None, index, period_ms

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          str(self.period_ms)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def load_framegen():
    """The synthetic frame generator WITHOUT the CUDA product library: fdreadoutlibs_b200/framegen.py binds only
    libswtpg_framegen.so and imports nothing else of the package, so it is loaded by path (the reference arm must not map
    libswtpg_b200.so)."""
    spec = importlib.util.spec_from_file_location("swtpg_framegen_standalone", os.path.join(ROOT, "fdreadoutlibs_b200", "framegen.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_reference_run(threshold: int, steps: int, warmup: int, pulse_rate: float):
    """The reference's own AVX2 SWTPG (oracle/_ref/libswtpg_ref.so: its headers compiled unmodified) on all host cores:
    expand_wibeth_adcs + process_window_avx2 + hit decode, one pinned worker per core, links dealt round-robin.
    Bounded sample: 8 links per core x 256 frames of the same synthetic workload. Returns (samples/s, dict)."""
    G = load_framegen()
    from oracle import binding as B

    cores = host_cores()
    kind = "reference" if B.reference_available() else "port"
    n_links, n_frames = 8 * cores, 256
    frames = G.gen_wibeth_host(G.gen_params(2, pulse_rate), n_links, n_frames, n_threads=cores)
    samples = n_links * n_frames * SAMPLES_PER_FRAME
    if kind == "reference":
        for _ in range(max(1, warmup)):
            B.ref_wibeth_bench(frames, cores, B.REF_ETH_SIMPLE_AVX2, threshold, 10, reps=1)
        secs = [B.ref_wibeth_bench(frames, cores, B.REF_ETH_SIMPLE_AVX2, threshold, 10, reps=1)[0] for _ in range(max(1, steps))]
    else:  # reference library not shipped: time the C restatement instead (single thread)
        cores = 1
        cfg = B.make_config(threshold=threshold)
        secs = []
        for _ in range(max(1, min(steps, 3))):
            t0 = time.perf_counter()
            B.oracle_process_links(cfg, frames)
            secs.append(time.perf_counter() - t0)
    total = sum(secs)
    value = samples * len(secs) / total
    extra = {}
    if kind == "reference":  # SURVEY 8(d): also one worker alone (per-core figure), AVX2 and the scalar "naive" processor
        one = frames[:8]
        t_avx = min(B.ref_wibeth_bench(one, 1, B.REF_ETH_SIMPLE_AVX2, threshold, 10, reps=1)[0] for _ in range(3))
        t_naive = B.ref_wibeth_bench(one[:2], 1, B.REF_ETH_SIMPLE_NAIVE, threshold, 10, reps=1)[0]
        per_core = 8 * n_frames * SAMPLES_PER_FRAME / t_avx
        extra = {"avx2_one_core": per_core, "naive_one_core": 2 * n_frames * SAMPLES_PER_FRAME / t_naive,
                 "links_real_time_per_core": per_core / 125.0e6, "us_per_frame_per_core": SAMPLES_PER_FRAME / per_core * 1e6,
                 "core_seconds_per_apa_second": APA_SAMPLES_PER_S / per_core}
    info = {"value": value, "unit": UNIT, "cores": cores, "kind": kind, **extra,
            "sample": f"{n_links} links x {n_frames} frames ({samples / 1e6:.0f} Msamples, {n_links * n_frames * FRAME_BYTES / 1e6:.0f} MB) per pass, "
                      f"{len(secs)} timed passes, threshold {threshold}, one pinned worker per core",
            "ms_per_pass": 1e3 * total / len(secs)}
    return value, info


CPU_KEYS = ("value", "unit", "cores", "kind", "sample", "avx2_one_core", "naive_one_core", "links_real_time_per_core", "us_per_frame_per_core",
            "core_seconds_per_apa_second")


class OneLineStdout:
    """Everything any library writes to fd 1 during the run (NCCL's version banner, the reference's setState printout, ...)
    goes to stderr; the JSON line is the only thing that reaches the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line: str):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


def bind_near_gpu(local_rank: int, world: int):
    """Pin this rank (and every thread it starts) to host cores next to its GPU: the cores of the GPU's NUMA node
    (/sys/bus/pci/devices/<bus id>/local_cpulist), shared evenly between the ranks whose GPUs sit on the same node. Returns what
    was done, for the record."""
    try:
        import torch

        allowed = sorted(os.sched_getaffinity(0))
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        domain = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        near = None
        if bus is not None:
            path = f"/sys/bus/pci/devices/{domain:04x}:{bus:02x}:{dev:02x}.0/local_cpulist"
            if os.path.exists(path):
                near = set()
                for part in open(path).read().strip().split(","):
                    if part:
                        a, _, b = part.partition("-")
                        near.update(range(int(a), int(b or a) + 1))
        cand = [c for c in allowed if near is None or c in near] or allowed
        if world > 1:  # ranks on the same node share it evenly; without topology information every rank gets its slice of all cores
            share = max(1, len(cand) // world) if near is None else max(1, len(cand) * 1 // max(1, min(world, 4)))
            start = (local_rank * share) % max(1, len(cand))
            mine = (cand + cand)[start:start + share]
        else:
            mine = cand
        os.sched_setaffinity(0, set(mine))
        return {"cores": len(mine), "numa_local": near is not None, "first_core": mine[0]}
    except Exception as e:  # binding is an optimisation, never a requirement
        return {"cores": host_cores(), "numa_local": False, "error": str(e)[:80]}


def main():
    out = OneLineStdout()
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    workload = (f"BASELINE config[2] per-GPU shard: {args.links} WIBEth links ({args.links / 40:.0f} APAs, {args.links * 64} channels) x "
                f"{args.frames} frames per step, synthetic noise+pulses, SimpleThreshold thr {args.threshold}")

    if args.impl == "reference":
        if rank != 0:
            return 0
        value, info = cpu_reference_run(args.threshold, args.steps, args.warmup, args.pulse_rate)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": info["ms_per_pass"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int16", "data": "synthetic",
                "config": {"workload": workload, "note": "reference arm: bounded sample of the same workload on the host cores"},
                "cpu_baseline": {k: info[k] for k in CPU_KEYS if k in info},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "real_time_apas": value / APA_SAMPLES_PER_S}
        out.emit(json.dumps(line))
        return 0

    import numpy as np
    import torch

    import fdreadoutlibs_b200 as S
    from fdreadoutlibs_b200 import frames as F
    from fdreadoutlibs_b200 import hostshim as H
    from fdreadoutlibs_b200 import sharding

    if not torch.cuda.is_available() or not S.device_available():
        print("bench.py: no CUDA device (this framework has no CPU fallback)", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    binding = bind_near_gpu(local_rank, world)

    n_links, frames = args.links, args.frames
    link0 = rank * n_links  # weak scaling: every rank owns its own block of links (global link numbers differ)
    nbytes = n_links * frames * FRAME_BYTES
    samples_per_step = n_links * frames * SAMPLES_PER_FRAME
    hbm_peak, peak_src = peaks()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # --- the checker: after a timed variant, reset the state, run ONE more launch on the same resident frames and compare the TPs of
    #     four sampled links with the CPU oracle (test infrastructure, never inside a timed region) ---
    def verify(g, d_tensor, fmt, algorithm, thr, links, units, unit_bytes, link_base=0, tp_cap=1 << 22, fir_taps=None):
        from oracle import binding as B

        g.stop()
        g.start()
        g.process_device(d_tensor.data_ptr(), units)
        got = g.fetch_tps(cap=tp_cap)
        sample = sorted({0, links // 3, (2 * links) // 3, links - 1})
        kw = {"fir_taps": fir_taps} if fir_taps is not None else {}
        cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS[algorithm], threshold=thr, **kw)
        view = d_tensor.view(links, units, unit_bytes)
        for l in sample:
            host = view[l].cpu().numpy()
            want = F.sort_tps(B.Oracle(cfg, link_id=l).process(host, cap=1 << 20))
            mine = F.sort_tps(got[got["link"] == l])
            if mine.size != want.size or not (mine == want).all():
                raise AssertionError(f"bench verification failed: {fmt} {algorithm} thr {thr}, link {link_base + l}: {mine.size} TPs, oracle {want.size}")
        return len(sample)

    # --- inputs resident in HBM before the timed region; 2.7 GB per step >> 126 MB L2, so no step re-reads from L2 ---
    d_frames = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    gp = S.gen_params(2, args.pulse_rate)
    S.gen_wibeth_device(gp, d_frames.data_ptr(), n_links, frames, link0=link0)
    torch.cuda.synchronize()

    gen = S.TPGenerator(n_links, frames, algorithm="SimpleThreshold", threshold=args.threshold, acc_limit=10, device=local_rank,
                        tp_capacity=1 << 22)
    gen.start()
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(max(3, args.warmup)):
        gen.process_device(d_frames.data_ptr(), frames, stream=stream)
    tps_per_step = gen.fetch_count()

    # --- timed region: exactly K steps, device time by CUDA events on the launching stream ---
    kernel_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for _ in range(args.steps):
            gen.process_device(d_frames.data_ptr(), frames, stream=stream)
        ev1.record()
        torch.cuda.synchronize()
        if args.dump_outputs and rank == 0:
            dump_tps(args.dump_outputs, gen.fetch_tps(cap=1 << 22))
        # long enough for nvidia-smi to see the load: repeat untimed launches for ~1 s, collecting per-launch times
        t_end = time.time() + 1.0
        while time.time() < t_end:
            gen.process_device(d_frames.data_ptr(), frames, stream=stream)
            kernel_ms.append(gen.last_kernel_ms())
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    local_ms_per_step = total_ms / args.steps
    tps_per_step = gen.fetch_count()
    ms_per_step = max_over_ranks(total_ms) / args.steps
    value = world * samples_per_step / (ms_per_step * 1e-3)
    verified_main = verify(gen, d_frames, "wibeth", "SimpleThreshold", args.threshold, n_links, frames, FRAME_BYTES, link_base=link0)

    # --- roofline of the fused kernel (rank-local): algorithmic bytes per launch / mean launch duration ---
    k_ms = local_ms_per_step
    algo_bytes = n_links * frames * FRAME_BYTES + tps_per_step * TP_BYTES + 2 * STATE_BYTES_PER_CHANNEL * n_links * 64
    achieved = algo_bytes / (k_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": None,
                "peak_source": peak_src, "kernel": "wibeth_kernel<PackedSimpleT<true>, 1 warp per CTA, ring 2 x 32 ticks> (software-pipelined policy, 20 persistent warps per SM, links handed out in 4 halving slices)", "kernel_ms": k_ms,
                "kernel_ms_per_launch_events": sum(kernel_ms) / len(kernel_ms), "algorithmic_bytes_per_launch": algo_bytes,
                "verified_links": verified_main}
    prof = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(prof):  # bytes per launch from the committed ncu --set full capture of this same workload
        with open(prof) as f:
            tr = json.load(f)
        if tr.get("links") == n_links and tr.get("frames") == frames:
            roofline["traffic"] = tr["dram_bytes_per_launch"]

    # =====================================================================================================================
    # e2e: the streaming plug-in path (every rank drives its own GPU at the same time)
    # =====================================================================================================================
    s_links, s_units, s_sc = args.stream_links, args.stream_units, 64
    feeders = max(1, min(args.feeders, binding["cores"]))
    lat_buf = S.gen_wibeth_host(gp, s_links, s_units, link0=link0, n_threads=max(1, min(8, binding["cores"])))  # the "latency buffer"
    warm = lat_buf[:, :128].copy()

    def run_stream(zero_copy, threads, passes, pace=0.0, n_slots=4, links=s_links, verify_links=0, all_ranks=False):
        buf = lat_buf[:links]
        with H.FrameProcessors(links, s_sc, threshold=args.threshold, device=local_rank, emulator_mode=False, block_on_backpressure=pace == 0,
                               count_only_sink=verify_links == 0, n_slots=n_slots, first_link_id=0) as fp:
            if zero_copy:  # the payload array plays the latency buffer the constframeptrs point into
                fp.register_buffer(buf)
            fp.start()
            fp.push_feeders(np.ascontiguousarray(warm[:links]), n_threads=threads, burst=16)  # staging ring allocation, first launches
            time.sleep(0.02)
            if all_ranks:  # every rank drives its own GPU at the same time (a collective: only where every rank makes this call)
                barrier()
            else:
                torch.cuda.synchronize()
            r0, t0 = resource.getrusage(resource.RUSAGE_SELF), time.perf_counter()
            st = fp.push_feeders(buf, n_threads=threads, burst=16, pace=pace, passes=passes)
            fp.stop()  # flush of the ragged tail, every remaining TriggerPrimitive delivered
            dt = time.perf_counter() - t0
            r1 = resource.getrusage(resource.RUSAGE_SELF)
            cpu_s = (r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)
            dropped = sum(fp.get_info(l)["num_frames_dropped_busy"] for l in range(links))
            cnt = fp.counters()
            tim = fp.stream_timing()
            n_tp = fp.tp_count()
            checked = 0
            if verify_links:  # untimed: the TriggerPrimitives of sampled links against the oracle (offline channel through the LUT, H2)
                from oracle import binding as B

                cfg = B.make_config(threshold=args.threshold)
                for l in sorted({0, links // 2, links - 1})[:verify_links]:
                    got = fp.take_tps(l, cap=1 << 20)
                    n_tp += got.size
                    seq = np.concatenate([warm[l]] + [buf[l]] * passes)
                    want = F.sort_tps(B.Oracle(cfg, link_id=l).process(seq, cap=1 << 20))
                    key = lambda a, ch: sorted(zip(a["time_start"].tolist(), ch, a["adc_integral"].tolist(), a["adc_peak"].tolist(),
                                                    a["time_over_threshold"].tolist()))
                    lut = np.array(fp.register_channel_map(l))
                    if key(got, got["channel"].tolist()) != key(want, lut[want["channel"]].tolist()):
                        raise AssertionError(f"bench verification failed: streaming path, link {l}: {got.size} TPs, oracle {want.size}")
                    checked += 1
            if zero_copy:
                fp.register_buffer(buf, on=False)
        n = passes * links * s_units
        return {"value": (n - dropped) * SAMPLES_PER_FRAME / dt, "unit": UNIT, "host_gbs": (n - dropped) * FRAME_BYTES / dt / 1e9, "wall_seconds": dt,
                "links": links, "feeder_threads": threads, "superchunk_frames": s_sc, "frames": n, "frames_dropped": dropped,
                "host_cores_busy": cpu_s / dt, "feeder_cores_busy": st["feeder_cpu_s"] / dt, "feeder_us_per_frame": st["feeder_cpu_s"] / n * 1e6,
                "core_seconds_per_apa_second": (cpu_s / dt) / max(1e-9, (n - dropped) * SAMPLES_PER_FRAME / dt / APA_SAMPLES_PER_S),
                "units_by_address": cnt["units_zero_copy"], "units_by_copy": cnt["units_staged"], "batches": cnt["batches"], "tps": n_tp,
                "late_bursts": st["late_bursts"], "verified_links": checked,
                # device time of the engine's batches (CUDA events): the gather kernel IS the host-link transfer
                "gather_ms_per_batch": tim["gather_ms"] / max(1, tim["batches"]), "kernel_ms_per_batch": tim["kernel_ms"] / max(1, tim["batches"]),
                "gather_gbs_while_active": cnt["h2d_bytes"] / max(1e-9, tim["gather_ms"]) / 1e6}

    stream_main = run_stream(True, feeders, args.stream_passes, all_ranks=True)
    e2e_dt = max_over_ranks(stream_main["wall_seconds"])
    e2e_frames = sum_over_ranks(stream_main["frames"] - stream_main["frames_dropped"])
    e2e_value = e2e_frames * SAMPLES_PER_FRAME / e2e_dt
    batches = max(1, stream_main["batches"])
    e2e = {"value": e2e_value, "unit": UNIT,
           "h2d_bytes_per_step": int((stream_main["frames"] - stream_main["frames_dropped"]) * FRAME_BYTES / batches),
           "d2h_bytes_per_step": int(stream_main["tps"] * TP_BYTES / batches) + 4,
           "step": "one dispatched batch of the streaming path (ragged, up to 64 frames per link)", "steps": batches,
           "path": "WIBEthFrameProcessor::find_hits -> swtpg_submit (zero-copy from the registered latency buffer) -> gather kernel over the host link -> "
                   "fused TPG kernel -> TP list to pinned host memory -> TriggerPrimitives to the tp_out sinks",
           "h2d_gbs_per_gpu": stream_main["host_gbs"], "real_time_apas": e2e_value / APA_SAMPLES_PER_S,
           "host_cores_busy_per_gpu": stream_main["host_cores_busy"], "feeder_threads_per_gpu": feeders, "links_per_gpu": s_links,
           "core_seconds_per_apa_second": stream_main["core_seconds_per_apa_second"],
           "reference_core_seconds_per_apa_second": REF_US_PER_FRAME_PER_CORE * 1e-6 * 40 * 62.5e6 / 2048,
           "ms_per_step": e2e_dt * 1e3 / batches}

    # --- e2e_batch: the batch entry point from one pinned buffer, and the host link's own ceiling measured with every rank copying at once ---
    wc = os.environ.get("SWTPG_BENCH_WC", "0") != "0"
    h_buf = S.PinnedBuffer(nbytes, write_combined=wc)
    h_frames = torch.from_numpy(h_buf.array)
    h_frames.copy_(d_frames)
    torch.cuda.synchronize()
    h_np = h_buf.array.reshape(n_links, frames, FRAME_BYTES)
    tp_cap = 1 << 22
    h_tps = torch.empty(tp_cap * TP_BYTES, dtype=torch.uint8, pin_memory=True).numpy().view(S.frames.TP_DTYPE)
    h2d_ms = []
    for _ in range(3):  # plain pinned copy of the same buffer, ALL ranks at the same time (barrier first): the platform's concurrent ceiling
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        d_frames.copy_(h_frames, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        h2d_ms.append(c0.elapsed_time(c1))
    h2d_peak_gbs = nbytes / (max_over_ranks(min(h2d_ms)) * 1e-3) / 1e9
    gen.stop()
    gen.start()
    n_tp = 0
    for _ in range(2):
        n_tp = gen.process_host(h_np, out=h_tps).size
    barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        n_tp = gen.process_host(h_np, out=h_tps).size
    torch.cuda.synchronize()
    b_s = max_over_ranks((time.perf_counter() - t0) / 4)
    e2e_batch = {"value": world * samples_per_step / b_s, "unit": UNIT, "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": n_tp * TP_BYTES + 4,
                 "ms_per_step": b_s * 1e3, "h2d_gbs_per_gpu": nbytes / b_s / 1e9, "real_time_apas": world * samples_per_step / b_s / APA_SAMPLES_PER_S,
                 "path": "swtpg_process_host: one pinned buffer of 5920 links x 64 frames, one copy, kernel, TP list back",
                 "ingest_roofline": {"bound": "host link (H2D)", "achieved": nbytes / b_s / 1e9, "peak": h2d_peak_gbs, "unit": "GB/s",
                                     "frac": (nbytes / b_s / 1e9) / h2d_peak_gbs,
                                     "peak_source": f"plain pinned H2D copy of the same buffer, all {world} rank(s) copying at the same time behind a barrier "
                                                    "(best of 3, slowest rank)"}}
    e2e["ingest_roofline"] = {"bound": "host link (H2D)", "achieved": stream_main["host_gbs"], "peak": h2d_peak_gbs, "unit": "GB/s",
                              "frac": stream_main["host_gbs"] / h2d_peak_gbs, "peak_source": e2e_batch["ingest_roofline"]["peak_source"]}
    del h_frames, h_np
    h_buf.close()

    # --- BASELINE config[2] as written: the module's links SPLIT over the GPUs (strong scaling), each rank's TP list ordered on the host
    #     and merged on rank 0 in time order (what TPCTPRequestHandler consumes) ---
    m_link0, m_n = sharding.shard_links(args.module_links, world, rank)
    d_m = torch.empty(m_n * frames * FRAME_BYTES, dtype=torch.uint8, device="cuda")
    S.gen_wibeth_device(gp, d_m.data_ptr(), m_n, frames, link0=m_link0)
    torch.cuda.synchronize()
    with S.TPGenerator(m_n, frames, threshold=args.threshold, device=local_rank, tp_capacity=1 << 22, sorted_tps=True) as g:
        g.start()
        for _ in range(3):
            g.process_device(d_m.data_ptr(), frames)
        g.fetch_count()
        barrier()
        ms = []
        for _ in range(10):
            g.process_device(d_m.data_ptr(), frames)
            g.fetch_count()
            ms.append(g.last_kernel_ms())
        shard_ms = max_over_ranks(sum(ms) / len(ms))
        # the rank's TP list, ordered by (time_start, link, channel) ON THE DEVICE before it crosses the host link (SWTPG_FLAG_SORTED_TPS)
        dev_sort = []
        for _ in range(3):
            g.process_device(d_m.data_ptr(), frames)
            mine = g.fetch_tps(cap=1 << 22)
            dev_sort.append(g.sort_stats()["last_ms"])
        dev_sort_ms = max_over_ranks(min(dev_sort))
        mine = sharding.globalise(mine, m_link0)
        # what the same ordering costs on one host core (round 1's path), on a shuffled copy; also the check of the device's order
        shuffled = mine[np.random.default_rng(5).permutation(mine.size)]
        t0 = time.perf_counter()
        by_host = S.sort_tps(shuffled)
        sort_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        if not (by_host == mine).all() or g.sort_stats()["finished_on_host"] != 0:
            raise AssertionError("device-ordered TP list differs from the host's ordering")
        del shuffled, by_host
        merged_n, merge_ms, transport_ms = mine.size, 0.0, 0.0
        if dist is not None:
            barrier()
            sharding.gather_and_merge(mine)  # untimed: the first collective of a shape pays for the communicator's set-up
            barrier()
            tm = {}
            merged = sharding.gather_and_merge(mine, timings=tm)  # host side: rank 0 receives the sorted lists and merges them
            merge_ms, transport_ms = tm.get("merge_s", 0.0) * 1e3, tm.get("gather_s", 0.0) * 1e3
            if rank == 0:
                merged_n = merged.size
                ok = bool((merged["time_start"][1:] >= merged["time_start"][:-1]).all())
                if not ok:
                    raise AssertionError("merged TP list is not time-ordered")
        v_strong = verify(g, d_m, "wibeth", "SimpleThreshold", args.threshold, m_n, frames, FRAME_BYTES, link_base=m_link0)
    by = m_n * frames * FRAME_BYTES + mine.size * TP_BYTES + 2 * STATE_BYTES_PER_CHANNEL * m_n * 64
    strong = {"workload": f"BASELINE config[2] as written: {args.module_links} links ({args.module_links / 40:.0f} APAs) split over {world} GPU(s), "
                          f"{m_n} links on this one, {frames} frames per step, resident in HBM", "links_per_gpu": m_n, "kernel_ms": shard_ms,
              "value": args.module_links * frames * SAMPLES_PER_FRAME / (shard_ms * 1e-3), "unit": UNIT,
              "real_time_apas": args.module_links * frames * SAMPLES_PER_FRAME / (shard_ms * 1e-3) / APA_SAMPLES_PER_S,
              "real_time_multiple_of_the_module": args.module_links * frames * SAMPLES_PER_FRAME / (shard_ms * 1e-3) / (args.module_links / 40 * APA_SAMPLES_PER_S),
              "roofline_frac_per_gpu": by / (shard_ms * 1e-3) / 1e9 / hbm_peak, "tps_per_step_per_gpu": int(mine.size),
              "device_sort_ms": dev_sort_ms, "host_sort_ms_per_gpu": sort_ms, "merge_ms": merge_ms, "gather_to_rank0_ms": transport_ms, "merged_tps": int(merged_n), "verified_links": v_strong,
              "merge": "each rank's list comes back ordered by (time_start, link, channel), ordered on the device (SWTPG_FLAG_SORTED_TPS: an LSD radix "
                       "sort of packed keys in HBM = device_sort_ms; host_sort_ms_per_gpu = the same ordering by swtpg_sort_tps on one host core, "
                       "for comparison, and the two lists are asserted identical); rank 0 receives the ordered lists (gather_to_rank0_ms: torch.distributed "
                       "all_gather of the lists as byte tensors, device-to-device under NCCL, + one copy to the host; bench plumbing — in a readout "
                       "application the lists arrive over its own network layer) and merges them with a k-way merge (swtpg_merge_sorted = "
                       "merge_ms): no collective inside the TPG path itself"}
    del d_m

    # --- BASELINE config[1]: ONE APA (40 links) on one GPU, and the shards of config[2] at 8 / 4 / 2 GPUs: launches that cannot fill a GPU ---
    single = None
    sweep = None
    if rank == 0:
        sl, sf = 40, 2048
        d1 = torch.empty(sl * sf * FRAME_BYTES, dtype=torch.uint8, device="cuda")
        S.gen_wibeth_device(gp, d1.data_ptr(), sl, sf)
        torch.cuda.synchronize()
        with S.TPGenerator(sl, sf, threshold=args.threshold, device=local_rank, tp_capacity=1 << 21) as g1:
            g1.start()
            ms1 = []
            for _ in range(4):
                g1.process_device(d1.data_ptr(), sf)
                g1.fetch_count()
                ms1.append(g1.last_kernel_ms())
            s1 = sl * sf * SAMPLES_PER_FRAME / (min(ms1[1:]) * 1e-3)
            v1 = verify(g1, d1, "wibeth", "SimpleThreshold", args.threshold, sl, sf, FRAME_BYTES, tp_cap=1 << 21)
            single = {"workload": "BASELINE config[1]: one APA = 40 links x 2048 frames resident in HBM", "value": s1, "unit": UNIT,
                      "kernel_ms": min(ms1[1:]), "real_time_multiple": s1 / APA_SAMPLES_PER_S, "verified_links": v1}
        del d1
        sweep = {}
        for links in (240, 750, 1500, 3000):
            with S.TPGenerator(links, frames, threshold=args.threshold, device=local_rank, tp_capacity=1 << 21) as g:
                g.start()
                ms = []
                for _ in range(8):
                    g.process_device(d_frames.data_ptr(), frames)  # the first `links` links of the resident batch
                    ntp = g.fetch_count()
                    ms.append(g.last_kernel_ms())
                k = min(ms[2:])
                by = links * frames * FRAME_BYTES + ntp * TP_BYTES + 2 * STATE_BYTES_PER_CHANNEL * links * 64
                sweep[str(links)] = {"kernel_ms": k, "value": links * frames * SAMPLES_PER_FRAME / (k * 1e-3), "roofline_frac": by / (k * 1e-3) / 1e9 / hbm_peak}

    # --- the other kernels of the path, same box, same run (rank 0): FIR + IQR, running sums, WIB2, high-occupancy stress ---
    others = None
    if rank == 0 and not args.no_variants:
        others = {}

        def timed(fmt, algorithm, thr, d_tensor, links, units, unit_bytes, samples_per_unit, state_bytes, tp_cap=1 << 22, fir_taps=None, check=True):
            with S.TPGenerator(links, units, fmt=fmt, algorithm=algorithm, threshold=thr, device=local_rank, tp_capacity=tp_cap,
                               fir_taps=fir_taps) as g:
                g.start()
                for _ in range(3):
                    g.process_device(d_tensor.data_ptr(), units)
                g.fetch_count()
                ms = []
                for _ in range(5):
                    g.process_device(d_tensor.data_ptr(), units)
                    ntp = g.fetch_count()
                    ms.append(g.last_kernel_ms())
                k = sum(ms) / len(ms)
                v = verify(g, d_tensor, fmt, algorithm, thr, links, units, unit_bytes, tp_cap=tp_cap, fir_taps=fir_taps) if check else 0
                by = links * units * unit_bytes + ntp * TP_BYTES + 2 * state_bytes * links * (256 if fmt == "wib2" else 64)
                return {"value": links * units * samples_per_unit / (k * 1e-3), "unit": UNIT, "kernel_ms": k, "tps_per_step": ntp, "verified_links": v,
                        "roofline": {"bound": "hbm", "achieved": by / (k * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                     "frac": by / (k * 1e-3) / 1e9 / hbm_peak}}

        # BASELINE config[1]/[2] data already resident (SimpleThreshold workload): FIR + IQR matched filter, AbsRS, StandardRS
        others["wibeth_fir_iqr_thr5"] = timed("wibeth", "FIR", 5, d_frames, n_links, frames, FRAME_BYTES, SAMPLES_PER_FRAME, 38)
        # taps other than firwin_int(7, 0.1, 64): the packed multiply-add policy (here firwin_int's taps at multiplier 32, doubled)
        others["wibeth_fir_iqr_other_taps"] = timed("wibeth", "FIR", 5, d_frames, n_links, frames, FRAME_BYTES, SAMPLES_PER_FRAME, 38,
                                                    fir_taps=[2, 6, 16, 20, 16, 6, 2])
        others["wibeth_abs_rs"] = timed("wibeth", "AbsRS", args.threshold, d_frames, n_links, frames, FRAME_BYTES, SAMPLES_PER_FRAME, 22)
        others["wibeth_standard_rs"] = timed("wibeth", "StandardRS", args.threshold, d_frames, n_links, frames, FRAME_BYTES, SAMPLES_PER_FRAME, 22)
        # BASELINE config[3]: high-occupancy stress — threshold 8 ADC (1.6 sigma), dense pulses
        S.gen_wibeth_device(S.gen_params(4, 0.5), d_frames.data_ptr(), n_links, frames, link0=link0)
        torch.cuda.synchronize()
        others["wibeth_simple_stress_thr8"] = timed("wibeth", "SimpleThreshold", 8, d_frames, n_links, frames, FRAME_BYTES, SAMPLES_PER_FRAME, 14,
                                                    tp_cap=1 << 27)
        # BASELINE config[4]: legacy WIB2 superchunks (256 channels x 12 ticks), SimpleThreshold and FIR + IQR
        w_links, w_units = n_links // 4, 340
        d_w = torch.empty(w_links * w_units * 5664, dtype=torch.uint8, device="cuda")
        S.gen_wib2_device(gp, d_w.data_ptr(), w_links, w_units)
        torch.cuda.synchronize()
        others["wib2_simple"] = timed("wib2", "SimpleThreshold", args.threshold, d_w, w_links, w_units, 5664, 256 * 12, 10)
        others["wib2_fir_iqr_thr5"] = timed("wib2", "FIR", 5, d_w, w_links, w_units, 5664, 256 * 12, 38)
        others["wib2_abs_rs"] = timed("wib2", "AbsRS", args.threshold, d_w, w_links, w_units, 5664, 256 * 12, 24)
        del d_w

    # --- more of the plug-in path (rank 0): against the clock at the detector's rate, with fewer feeders, with the copy-on-submit default ---
    plugin = None
    if rank == 0 and not args.no_variants:
        plugin = {"zero_copy": {k: v for k, v in stream_main.items()},
                  "zero_copy_2_feeders": run_stream(True, min(2, feeders), args.stream_passes),
                  "copy_on_submit_8_feeders": run_stream(False, min(8, binding["cores"]), max(2, args.stream_passes // 2)),
                  "paced_x1_200_links": run_stream(True, feeders, args.stream_passes, pace=1.0, n_slots=4, links=min(200, s_links)),
                  "paced_x1_240_links": run_stream(True, feeders, args.stream_passes, pace=1.0, n_slots=4),
                  "verification": run_stream(True, min(2, feeders), 1, links=min(40, s_links), verify_links=3),
                  "reference_us_per_frame_per_core": REF_US_PER_FRAME_PER_CORE,
                  "note": "zero_copy: the latency buffer is registered (swtpg_register_buffer) and find_hits hands over addresses; copy_on_submit: the "
                          "ABI's default for unregistered memory, every frame copied into the pinned staging ring by its feeder thread; paced_x1: "
                          "frames arrive at the detector's rate (one per link per 32.768 us) and submit never blocks — frames_dropped counts what a "
                          "full ring refused; host_cores_busy = user + system CPU time of the whole process (feeders, the library's dispatcher / "
                          "release / completion threads, the shim's delivery thread) over the wall time; the reference spends "
                          f"{REF_US_PER_FRAME_PER_CORE} us of one core per frame = {REF_US_PER_FRAME_PER_CORE * 1e-6 * 40 * 62.5e6 / 2048:.2f} core-seconds per "
                          "APA-second on the computation alone"}
    del lat_buf

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, range(os.cpu_count() or 1)) if hasattr(os, "sched_setaffinity") else None
        _, cpu = cpu_reference_run(args.threshold, steps=5, warmup=1, pulse_rate=args.pulse_rate)
        cpu = {k: cpu[k] for k in CPU_KEYS if k in cpu}

    gen.close()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16",
            "data": "synthetic",
            "config": {"workload": workload, "links_per_gpu": n_links, "frames_per_step": frames, "bytes_per_step_per_gpu": nbytes,
                       "l2_policy": "inputs larger than L2 (2.7 GB per step vs 126 MB)", "tps_per_step_per_gpu": tps_per_step,
                       "parallelism": f"links sharded over {world} GPU(s), no collective", "host_binding": binding},
            "real_time_apas": value / APA_SAMPLES_PER_S,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "e2e_batch": e2e_batch,
            "module_split": strong,
            "single_apa": single,
            "link_count_sweep": sweep,
            "other_kernels": others,
            "plugin_streaming": plugin,
            "gpu_launches": args.steps,
            "clocks": clocks.summary(),
        }
        out.emit(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

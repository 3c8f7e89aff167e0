"""Cost of the per-link channel covariance (SWTPG_FLAG_CHANNEL_COVARIANCE) on one GPU: the same handle with the flag off and on.

With the flag, every batch is read a second time, by the channel products kernel after its TPG kernel, on the same stream. The
kernel sums the products of every pair of a link's channels on the integer tensor cores (mma.sync m16n8k32 u8 x u8 -> s32 on byte
planes of the samples): 144 IMMA instructions per WIBEth frame, 396 per WIB2 superchunk (the launch sizes below give whole
slabs). On frames resident in HBM that work is what the flag costs; on the streaming path the host link bounds a step.

Resident-frame workloads (frames generated on the device: 64 units per link, threshold 60, 0.02 pulses per channel and 64 ticks):
WIBEth SimpleThreshold at 5920 links (the bench workload) and at 240 links (the streaming path's size), WIB2 SimpleThreshold at
1480 links. The two variants alternate round by round; each round times `--launches` back-to-back batches with CUDA events on the
launching stream. Reported per variant: median ms per batch, the range over rounds and Tsamples/s; for the flag on also the
IMMA instructions per batch and their rate over the added time (on - off), with the dense integer operations that makes
(16 x 8 x 32 multiply-adds, 2 operations each, per IMMA).

Streaming workload: 240 WIBEth links through the host shim's WIBEthFrameProcessors (push_feeders, 8 feeder threads, zero-copy from
a registered latency buffer of 1024 frames per link), flag off and on alternating; reported in GB/s of frames.

The card's name and power limit are read in the same run. Writes one JSON document to --out.

    python tools/channel_covariance_probe.py --out profiles/channel_covariance_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [("wibeth", 5920), ("wibeth", 240), ("wib2", 1480)]
# IMMA instructions per unit of one link (channel_products_kernel): a WIBEth frame is one diagonal 64 x 64 block over two K-steps
# of 32 ticks, 32 tiles of HL and 20 tiles touching the upper triangle of HH and LL; a WIB2 superchunk is 1/8 of a 96-tick slab
# of 4 diagonal blocks (3 K-steps x 72) and 6 off-diagonal blocks (3 K-steps x 32 tiles x 4 terms)
IMMA_PER_UNIT = {"wibeth": 2 * (32 + 2 * 20), "wib2": (4 * 3 * (32 + 2 * 20) + 6 * 3 * 32 * 4) // 8}
IMMA_OPS = 16 * 8 * 32 * 2
VARIANTS = {"flag off": False, "flag on": True}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"nvidia-smi failed: {e}"
    return out


def measure_resident(fmt, n_links, units, rounds, launches):
    import torch

    import fdreadoutlibs_b200 as S
    from fdreadoutlibs_b200 import frames as F

    wib2 = fmt == "wib2"
    unit_bytes, channels = (F.WIB2_SUPERCHUNK_BYTES, 256) if wib2 else (F.WIBETH_FRAME_BYTES, 64)
    samples = n_links * units * (12 if wib2 else 64) * channels
    d_frames = torch.empty(n_links * units * unit_bytes, dtype=torch.uint8, device="cuda")
    (S.gen_wib2_device if wib2 else S.gen_wibeth_device)(S.gen_params(2, 0.02), d_frames.data_ptr(), n_links, units)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    gens = {}
    for name, on in VARIANTS.items():
        g = S.TPGenerator(n_links, units, fmt=fmt, threshold=60, acc_limit=10, tp_capacity=1 << 22, channel_covariance=on)
        g.start()
        for _ in range(5):  # warm-up: module loads, occupancy queries
            g.process_device(d_frames.data_ptr(), units, stream=stream)
        gens[name] = [g, g.fetch_count(), []]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):  # alternate the variants
        for name, (g, _, ms) in gens.items():
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(launches):
                g.process_device(d_frames.data_ptr(), units, stream=stream)
            ev1.record()
            torch.cuda.synchronize()
            ms.append(ev0.elapsed_time(ev1) / launches)
    out = {}
    for name, (g, tps, ms) in gens.items():
        med = sorted(ms)[len(ms) // 2]
        out[name] = {"ms_per_batch": med, "ms_min": min(ms), "ms_max": max(ms), "tsamples_per_s": samples / (med * 1e-3) / 1e12,
                     "tps_per_batch": tps, "rounds": len(ms)}
        if name == "flag on":
            out[name]["tpg_kernel_ms_last"] = g.last_kernel_ms()
        g.close()
    imma = n_links * units * IMMA_PER_UNIT[fmt]
    added = (out["flag on"]["ms_per_batch"] - out["flag off"]["ms_per_batch"]) * 1e-3
    out["flag on"]["imma_per_batch"] = imma
    out["flag on"]["imma_per_s_over_added_time"] = imma / added if added > 0 else None
    out["flag on"]["int_tops_over_added_time"] = imma * IMMA_OPS / added / 1e12 if added > 0 else None
    del d_frames
    torch.cuda.empty_cache()
    return out


def measure_streaming(n_links, units, rounds, passes):
    import fdreadoutlibs_b200 as S
    from fdreadoutlibs_b200 import hostshim as H

    frames = S.gen_wibeth_host(S.gen_params(2, 0.02), n_links, units, n_threads=8)
    res = {name: [] for name in VARIANTS}
    for _ in range(rounds):
        for name, on in VARIANTS.items():
            with H.FrameProcessors(n_links, 64, threshold=60, n_slots=3, count_only_sink=True, channel_covariance=on) as fp:
                fp.register_buffer(frames)
                fp.start()
                fp.push_feeders(frames[:, :128].copy(), n_threads=8, burst=16)  # warm-up: engine creation, first launches
                t0 = time.perf_counter()
                st = fp.push_feeders(frames, n_threads=8, burst=16, passes=passes)
                fp.stop()
                dt = time.perf_counter() - t0
                fp.register_buffer(frames, on=False)
            res[name].append(st["payloads"] * frames.shape[2] / dt / 1e9)
    return {name: {"gb_per_s": sorted(v)[len(v) // 2], "gb_per_s_min": min(v), "gb_per_s_max": max(v), "rounds": len(v)}
            for name, v in res.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=50, help="launches per variant and round (at least 200 for 240 links)")
    ap.add_argument("--stream-rounds", type=int, default=3)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("channel_covariance_probe needs a GPU")
    doc = {"card": card(), "device": torch.cuda.get_device_name(0), "units_per_link": 64, "rounds": args.rounds,
           "launches_per_round": args.launches}
    for fmt, n in WORKLOADS:
        launches = args.launches if n > 240 else max(args.launches, 200)
        doc[f"{fmt} SimpleThreshold {n} links"] = measure_resident(fmt, n, 64, args.rounds, launches)
    doc["streaming shim 240 links zero-copy"] = measure_streaming(240, 1024, args.stream_rounds, 4)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(doc["card"])
    for key, r in doc.items():
        if not isinstance(r, dict):
            continue
        if "ms_per_batch" in r["flag off"]:
            base = r["flag off"]["ms_per_batch"]
            for name, v in r.items():
                print(f"{key:>34} | {name:<8} | {v['ms_per_batch']:.4f} ms ({v['ms_min']:.4f}-{v['ms_max']:.4f}) | "
                      f"{100 * (v['ms_per_batch'] / base - 1):+.2f} % | {v['tsamples_per_s']:.3f} Tsamples/s")
            if r["flag on"]["int_tops_over_added_time"]:
                print(f"{key:>34} | {r['flag on']['imma_per_batch']} IMMA per batch, {r['flag on']['imma_per_s_over_added_time']:.3e} IMMA/s "
                      f"= {r['flag on']['int_tops_over_added_time']:.1f} dense int8 Tops/s over the added time")
        else:
            for name, v in r.items():
                print(f"{key:>34} | {name:<8} | {v['gb_per_s']:.2f} GB/s ({v['gb_per_s_min']:.2f}-{v['gb_per_s_max']:.2f})")


if __name__ == "__main__":
    main()

"""Cost of per-channel threshold tables (swtpg_set_link_thresholds) on one GPU: the same handle with and without a table on every
link. A packed policy forms its comparison constant from the link's SV_THRESHOLD row once per work item (one 128-byte row read
and one clamp per 64-channel group), whether or not the link has a table, so "no tables" already pays for the row; what this
measures is that the kernel time does not depend on the tables.

Variants, all on frames resident in HBM (generated on the device; the bench's input: 64 units per link, threshold 60, 0.02
pulses per channel and 64 ticks), per workload:
  a  no tables
  b  every link with a table whose entries all equal the configuration's 60 (the same TPs as a)
  c  every link with its own table of thresholds 45..75 by channel (about the same hit count; different TPs)
Workloads: WIBEth SimpleThreshold at 5920 links (the bench workload) and 240 links (the streaming path's size), AbsRS and
StandardRS at 5920 links, WIB2 SimpleThreshold at 1480 links (as many channels as 5920 WIBEth links).

The variants of one workload alternate round by round; each round times `--launches` back-to-back launches with CUDA events on
the launching stream. Reported per variant: median ms per batch, the range over rounds and Tsamples/s. The card's name and
power limit are read in the same run. Writes one JSON document to --out.

    python tools/channel_threshold_probe.py --out profiles/channel_threshold_probe.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [("wibeth", "SimpleThreshold", 5920), ("wibeth", "SimpleThreshold", 240), ("wibeth", "AbsRS", 5920),
             ("wibeth", "StandardRS", 5920), ("wib2", "SimpleThreshold", 1480)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"nvidia-smi failed: {e}"
    return out


def measure(fmt, algorithm, n_links, units, rounds, launches):
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
    rng = np.random.default_rng(7)
    variants = {"a no tables": None,
                "b all-equal tables (60)": lambda l: np.full(channels, 60, dtype=np.uint16),
                "c own table per link (45..75)": lambda l: rng.integers(45, 76, channels).astype(np.uint16)}
    gens = {}
    for name, make in variants.items():
        g = S.TPGenerator(n_links, units, fmt=fmt, algorithm=algorithm, threshold=60, acc_limit=10, tp_capacity=1 << 22)
        if make is not None:
            for l in range(n_links):
                g.set_link_thresholds(l, make(l))
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
        g.close()
    del d_frames
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=50, help="launches per variant and round (at least 200 for 240 links)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("channel_threshold_probe needs a GPU")
    doc = {"card": card(), "device": torch.cuda.get_device_name(0), "units_per_link": 64, "rounds": args.rounds,
           "launches_per_round": args.launches}
    for fmt, algorithm, n in WORKLOADS:
        launches = args.launches if n > 240 else max(args.launches, 200)
        doc[f"{fmt} {algorithm} {n} links"] = measure(fmt, algorithm, n, 64, args.rounds, launches)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(doc["card"])
    for fmt, algorithm, n in WORKLOADS:
        key = f"{fmt} {algorithm} {n} links"
        base = doc[key]["a no tables"]["ms_per_batch"]
        for name, r in doc[key].items():
            print(f"{key:>34} | {name:<30} | {r['ms_per_batch']:.4f} ms ({r['ms_min']:.4f}-{r['ms_max']:.4f}) | "
                  f"{100 * (r['ms_per_batch'] / base - 1):+.2f} % | {r['tsamples_per_s']:.3f} Tsamples/s | {r['tps_per_batch']} TPs")


if __name__ == "__main__":
    main()

"""Cost of per-link TPG configurations (swtpg_set_link_config) on one GPU: the batch kernel runs once per configuration group,
the groups one after another on one stream.

Variants, all on frames resident in HBM (generated on the device; the bench's input: 64 frames per link, threshold 60,
0.02 pulses per channel and 64 ticks):
  5920 links (the bench workload)
    a  uniform SimpleThreshold handle
    b  the same handle with every link set to the handle's own configuration (one group: must time as a)
    c  two thresholds interleaved by link (2 groups of 2960)
    d  six thresholds interleaved by link (6 groups)
    e  half SimpleThreshold, half AbsRS (2 groups)
  240 links (the streaming path's size): 1, 2 and 6 groups (thresholds interleaved by link)

The variants of one size alternate round by round; each round times `--launches` back-to-back launches with CUDA events on the
launching stream. Reported per variant: median ms per batch (and the range over rounds), Tsamples/s, and the share of the HBM
peak in bench.py's accounting (frames read once + TP records + carried state in and out). The card's name and power limit are
read in the same run. Writes one JSON document to --out.

    python tools/link_config_probe.py --out profiles/r03_link_config_probe.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FRAME_BYTES, SAMPLES_PER_FRAME, TP_BYTES, STATE_BYTES_PER_CHANNEL = 7200, 64 * 64, 32, 14  # as bench.py
DESIGN_PEAK_GBS = 6452.5  # the HBM peak DESIGN.md quotes


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return DESIGN_PEAK_GBS, "DESIGN.md's 6452.5 GB/s (no MEASURED_PEAKS.json on this machine)"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"nvidia-smi failed: {e}"
    return out


def variants_for(n_links):
    """name -> {link: set_link_config kwargs} (None = no call at all)."""
    thr6 = (60, 40, 50, 70, 80, 90)
    if n_links == 240:
        return {"1 group": None,
                "2 groups (thresholds 60 / 40 by link)": {l: dict(threshold=(60, 40)[l % 2]) for l in range(n_links)},
                "6 groups (six thresholds by link)": {l: dict(threshold=thr6[l % 6]) for l in range(n_links)}}
    return {"a uniform": None,
            "b every link set to the handle's configuration": {l: {} for l in range(n_links)},
            "c 2 groups (thresholds 60 / 40 by link)": {l: dict(threshold=(60, 40)[l % 2]) for l in range(n_links)},
            "d 6 groups (six thresholds by link)": {l: dict(threshold=thr6[l % 6]) for l in range(n_links)},
            "e half SimpleThreshold, half AbsRS": {l: (dict(algorithm="AbsRS") if l % 2 else {}) for l in range(n_links)}}


def measure(n_links, frames, rounds, launches, peak):
    import torch

    import fdreadoutlibs_b200 as S

    d_frames = torch.empty(n_links * frames * FRAME_BYTES, dtype=torch.uint8, device="cuda")
    S.gen_wibeth_device(S.gen_params(2, 0.02), d_frames.data_ptr(), n_links, frames)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream().cuda_stream
    gens = {}
    for name, links in variants_for(n_links).items():
        g = S.TPGenerator(n_links, frames, threshold=60, acc_limit=10, tp_capacity=1 << 22)
        for l, kw in (links or {}).items():
            g.set_link_config(l, **kw)
        g.start()
        for _ in range(5):  # warm-up: module loads, occupancy queries
            g.process_device(d_frames.data_ptr(), frames, stream=stream)
        gens[name] = [g, g.fetch_count(), []]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):  # alternate the variants
        for name, (g, _, ms) in gens.items():
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(launches):
                g.process_device(d_frames.data_ptr(), frames, stream=stream)
            ev1.record()
            torch.cuda.synchronize()
            ms.append(ev0.elapsed_time(ev1) / launches)
    out = {}
    for name, (g, tps, ms) in gens.items():
        med = sorted(ms)[len(ms) // 2]
        algo_bytes = n_links * frames * FRAME_BYTES + tps * TP_BYTES + 2 * STATE_BYTES_PER_CHANNEL * n_links * 64
        out[name] = {"ms_per_batch": med, "ms_min": min(ms), "ms_max": max(ms), "tsamples_per_s": n_links * frames * SAMPLES_PER_FRAME / (med * 1e-3) / 1e12,
                     "hbm_frac": algo_bytes / (med * 1e-3) / 1e9 / peak, "tps_per_batch": tps, "rounds": len(ms)}
        g.close()
    del d_frames
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=50, help="launches per variant and round")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("link_config_probe needs a GPU")
    peak, peak_src = hbm_peak()
    doc = {"card": card(), "device": torch.cuda.get_device_name(0), "hbm_peak_gbs": peak, "peak_source": peak_src,
           "frames_per_link": 64, "rounds": args.rounds, "launches_per_round": args.launches,
           "5920 links": measure(5920, 64, args.rounds, args.launches, peak),
           "240 links": measure(240, 64, args.rounds, max(args.launches, 200), peak)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(f"{doc['card']}; HBM peak {peak} GB/s ({peak_src})")
    for size in ("5920 links", "240 links"):
        for name, r in doc[size].items():
            print(f"{size:>10} | {name:<48} | {r['ms_per_batch']:.4f} ms ({r['ms_min']:.4f}-{r['ms_max']:.4f}) | "
                  f"{r['tsamples_per_s']:.3f} Tsamples/s | {100 * r['hbm_frac']:.1f} % of HBM peak")


if __name__ == "__main__":
    main()

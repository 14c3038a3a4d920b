#!/usr/bin/env python
"""A/B timing of the spectrum export (fx_analyse_device_spectrum) against fx_analyse_device on a B200.

The bench workload (fx_synth_device: 4096 tracks x 10 s at 48 kHz, generated on the device) is analysed in the way bench.py
calls the engine (raw + smoothed outputs, no diagnostics, state carried from step to step), alternately with and without
the export, by one engine per spectrum mode, at N = 4096 / 2048 / 1024.  k_analyse is timed with fx_profile_enable /
fx_profile_read (CUDA events around each launch); each arm's median and spread over the timed steps are reported with the
extra HBM bytes the export writes and the card's name and power limit.  Writes one JSON document (--out; the measured ones
are kept under profiles/)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "feature-extractor_b200")]
import fxb200

SIZES = ((4096, 1024), (2048, 1024), (1024, 512))
MODES = {"re_squared": fxb200.SPECTRUM_RE_SQUARED, "power": fxb200.SPECTRUM_POWER}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    return [s.strip() for s in q.split(",")]


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=4096)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", required=True, help="JSON file to write")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures on the GPU only")
    sr, T = 48000.0, args.tracks
    name, power_limit, max_sm = card()
    report = {"gpu": name, "power_limit": power_limit, "max_sm_clock": max_sm, "tracks": T, "seconds": args.seconds,
              "steps": args.steps, "warmup": args.warmup, "timer": "fx_profile_read: CUDA events around k_analyse", "sizes": {}}
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    for N, H in SIZES:
        S = (int(sr * args.seconds) // H) * H
        F = S // H
        audio = torch.empty((T, S), dtype=torch.float32, device=dev)
        raw = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
        smooth = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
        spec = torch.empty((T, F, N // 2), dtype=torch.float32, device=dev)
        res = {"frames": T * F, "spec_bytes": spec.numel() * 4}
        for mode, v in MODES.items():
            e = fxb200.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=0, spectrum=v)
            e.synth_device(audio.data_ptr(), S, S, first_track=0, stream=sptr)
            torch.cuda.synchronize(dev)
            e.profile_enable(True)
            ms = {"plain": [], "export": []}
            for i in range(args.warmup + args.steps):
                order = ["plain", "export"] if i % 2 == 0 else ["export", "plain"]          # alternate which arm runs first
                for arm in order:
                    e.profile_read()
                    e.analyse_device(audio.data_ptr(), S, S, raw.data_ptr(), smooth.data_ptr(), None, stream=sptr,
                                     d_spec_ptr=spec.data_ptr() if arm == "export" else None)
                    torch.cuda.synchronize(dev)
                    k1, _, n = e.profile_read()
                    if i >= args.warmup:
                        ms[arm].append(k1)
            e.close()
            r = {arm: {"median_ms": statistics.median(x), "min_ms": min(x), "max_ms": max(x), "all_ms": x} for arm, x in ms.items()}
            r["export_over_plain"] = r["export"]["median_ms"] / r["plain"]["median_ms"] - 1.0
            r["extra_ms"] = r["export"]["median_ms"] - r["plain"]["median_ms"]
            res[mode] = r
            print(f"N={N} H={H} {mode}: k_analyse plain {r['plain']['median_ms']:.2f} ms [{r['plain']['min_ms']:.2f}, {r['plain']['max_ms']:.2f}], "
                  f"export {r['export']['median_ms']:.2f} ms [{r['export']['min_ms']:.2f}, {r['export']['max_ms']:.2f}]: "
                  f"{100 * r['export_over_plain']:+.2f} % ({r['extra_ms']:+.2f} ms for {res['spec_bytes'] / 1e9:.2f} GB)", flush=True)
        report["sizes"][f"N{N}_H{H}"] = res
        del audio, raw, smooth, spec
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(report, open(args.out, "w"), indent=1)
    print(name, power_limit)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""A/B timing of the two spectrum modes (fx_config.spectrum: the reference's Re(X)^2 and the power spectrum |X|^2) on a B200.

The bench workload (fx_synth_device: 4096 tracks x 10 s at 48 kHz, generated on the device) is analysed by two engines that
differ only in the mode, alternately in one process, in the way bench.py calls the engine (fx_analyse_device, raw + smoothed
outputs, no diagnostics, state carried from step to step).  k_analyse is timed with fx_profile_enable / fx_profile_read (CUDA
events around each launch); each mode's median and spread over the timed steps are reported with the card's name and power
limit.  Writes one JSON document (--out; the measured ones are kept under profiles/)."""
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
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
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
        engines = {m: fxb200.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=0, spectrum=v) for m, v in MODES.items()}
        audio = torch.empty((T, S), dtype=torch.float32, device=dev)
        raw = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
        smooth = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
        engines["re_squared"].synth_device(audio.data_ptr(), S, S, first_track=0, stream=sptr)
        torch.cuda.synchronize(dev)
        ms = {m: [] for m in MODES}
        for e in engines.values():
            e.profile_enable(True)
        for i in range(args.warmup + args.steps):
            order = list(MODES) if i % 2 == 0 else list(MODES)[::-1]          # alternate which mode runs first
            for m in order:
                e = engines[m]
                e.profile_read()
                e.analyse_device(audio.data_ptr(), S, S, raw.data_ptr(), smooth.data_ptr(), None, stream=sptr)
                torch.cuda.synchronize(dev)
                k1, _, n = e.profile_read()
                if i >= args.warmup:
                    ms[m].append(k1)
        for e in engines.values():
            e.close()
        del audio, raw, smooth
        torch.cuda.empty_cache()
        res = {m: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "all_ms": v} for m, v in ms.items()}
        res["power_over_re_squared"] = res["power"]["median_ms"] / res["re_squared"]["median_ms"] - 1.0
        res["frames"] = T * F
        report["sizes"][f"N{N}_H{H}"] = res
        print(f"N={N} H={H}: k_analyse re^2 {res['re_squared']['median_ms']:.2f} ms [{res['re_squared']['min_ms']:.2f}, {res['re_squared']['max_ms']:.2f}], "
              f"power {res['power']['median_ms']:.2f} ms [{res['power']['min_ms']:.2f}, {res['power']['max_ms']:.2f}]: "
              f"{100 * res['power_over_re_squared']:+.1f} %", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(report, open(args.out, "w"), indent=1)
    print(name, power_limit)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Per-config parity report, generated on the GPU box: the CUDA path through the C ABI against the reference's own classes
(oracle/_ref values, port margins -- tests/oracle_util.py::CheckedOracle) on every BASELINE.json config shape.  For each
config: frames, mismatching values, exempt values by cause (oracle-side decision margin < 1e-4), lag mismatches, frames only
the GPU flags as low-margin (diagnostic), and the largest absolute / relative error per feature over the values that were
compared numerically.  Writes one JSON document (default gpurun_out/parity.json; copied to profiles/parity_rNN.json)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "feature-extractor_b200"), os.path.join(ROOT, "tests")]
import fxb200
import oracle_util as ou
import power_oracle


def engine_offline(audio, N, H, sr, **kw):
    with fxb200.Engine(n_tracks=audio.shape[0], window=N, hop=H, sample_rate=sr, ring_hops=0, **kw) as e:
        return e.analyse_host(audio)


def engine_carried(audio, N, H, sr, calls):
    """the stream in `calls` consecutive fx_analyse_host calls, state carried"""
    T, S = audio.shape
    F = S // H
    cuts = [round(i * F / calls) * H for i in range(calls + 1)]
    parts = []
    with fxb200.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=0) as e:
        for a, b in zip(cuts[:-1], cuts[1:]):
            parts.append(e.analyse_host(audio[:, a:b]))
    return {k: np.concatenate([p[k] for p in parts], axis=1) for k in ("raw", "smooth", "diag")}


def engine_realtime(audio, N, H, sr, block, per_group):
    """through the pinned ring and the worker threads; smoothed rows only (what the real-time path publishes)"""
    T, S = audio.shape
    F = S // H
    smooth = np.zeros((T, F, 12), np.float32)
    with fxb200.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=8, tracks_per_group=per_group) as e:
        e.rt_start()
        for b0 in range(0, F * H, block):
            e.push_block(audio[:, b0:b0 + block])
            due = (b0 + block) // H
            if due != b0 // H:
                t0 = time.time()
                while True:
                    vec, idx = e.poll_block()
                    if (idx >= due).all():
                        break
                    if time.time() - t0 > 10:
                        raise RuntimeError(f"hop {due} never published")
                    time.sleep(0.0002)
                smooth[:, due - 1] = vec
        e.rt_stop()
    return smooth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "parity.json"))
    ap.add_argument("--quick", action="store_true", help="short streams (a smoke run of this script)")
    ap.add_argument("--spectrum", choices=("re2", "power"), default="re2",
                    help="power: only the configs[1] shape, the engine in power-spectrum mode (fx_config.spectrum = 1) against "
                         "tests/power_oracle.py")
    args = ap.parse_args()
    ora = ou.best_oracle() if args.spectrum == "re2" else power_oracle.CheckedPowerOracle()
    q = args.quick
    report = {"oracle": ora.kind, "tolerance": ou.TOL, "margin_tolerance": ou.MARGIN_TOL,
              "rule": "a mismatch is exempt only when the ORACLE's decision margin (port side) is below margin_tolerance; GPU margins are diagnostic",
              "spectrum": args.spectrum, "configs": {}}

    def add(name, what, g, o, extra=None):
        res = ou.compare(g, o)
        res["what"] = what
        res["exempt_frac_of_values"] = res["raw_mismatch_exempt"] / max(1, res["frames"] * 12)
        if extra:
            res.update(extra)
        report["configs"][name] = res
        print(name, ou.summary(res), flush=True)

    if args.spectrum == "power":
        # |X|^2 per bin (fx_engine.h FX_SPECTRUM_POWER) at the configs[1] shape: the one full-size leg of the mode
        N, H, sr = 2048, 512, 48000.0
        a = ou.make_tracks(8 if q else 64, (5 if q else 60) * 48000 // H * H, sr)
        add("c2_power", f"configs[1] shape in power-spectrum mode: {a.shape[0]} tracks x {a.shape[1] / sr:g} s, N=2048 H=512",
            engine_offline(a, N, H, sr, spectrum=fxb200.SPECTRUM_POWER), power_oracle.CheckedPowerOracle().analyse(a, window=N, hop=H, sample_rate=sr))
        c = report["configs"]["c2_power"]
        report["totals"] = {k: c[k] for k in ("frames", "raw_mismatch_total", "raw_mismatch_exempt", "bad_raw", "lag_mismatch", "bad_lag", "bad_smooth",
                                              "gpu_only_low_margin_frames", "exempt_by_cause", "max_abs_err")}
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        json.dump(report, open(args.out, "w"), indent=1)
        sys.exit(0 if c["bad_raw"] == 0 and c["bad_lag"] == 0 and c["bad_smooth"] == 0 else 1)

    # configs[0]: the reference's own CPU-runnable case, verbatim run() bodies (mode A)
    N, H, sr = 1024, 512, 44100.0
    a = ou.make_tracks(1, (441000 // H) * H, sr)
    add("c1", "configs[0]: 1 track, 44.1 kHz, 10 s, N=1024 H=512, oracle mode A", engine_offline(a, N, H, sr), ora.analyse(a, window=N, hop=H, sample_rate=sr, mode=0))

    # configs[1] in full
    N, H, sr = 2048, 512, 48000.0
    a = ou.make_tracks(8 if q else 64, (5 if q else 60) * 48000 // H * H, sr)
    add("c2", f"configs[1]: {a.shape[0]} tracks x {a.shape[1] / sr:g} s, N=2048 H=512", engine_offline(a, N, H, sr), ora.analyse(a, window=N, hop=H, sample_rate=sr))

    # configs[2] shape on the bench workload itself (Philox generator)
    N, H, sr = 4096, 1024, 48000.0
    a = ou.synth_tracks(16 if q else 128, (2 if q else 10) * 48000 // H * H, sr)
    add("c3", f"configs[2] shape: first {a.shape[0]} tracks x {a.shape[1] / sr:g} s of the bench workload, N=4096 H=1024",
        engine_offline(a, N, H, sr), ora.analyse(a, window=N, hop=H, sample_rate=sr))

    # configs[3]: the real-time path (pinned ring, worker threads), smoothed rows
    N, H, sr = 2048, 1024, 48000.0
    a = ou.synth_tracks(16 if q else 64, (3 if q else 20) * 48000 // H * H, sr)
    o = ora.analyse(a, window=N, hop=H, sample_rate=sr, mode=0)
    sm = engine_realtime(a, N, H, sr, 256, 16)
    off = engine_offline(a, N, H, sr)
    add("c4", f"configs[3] shape: {a.shape[0]} live tracks, 256-sample blocks, N=2048 H=1024, worker threads; raw / diag from the one-call analysis of the same stream, "
        "smoothed rows as published by the real-time path", {"raw": off["raw"], "diag": off["diag"], "smooth": sm}, o,
        {"realtime_rows_bit_identical_to_offline": bool(np.array_equal(sm, off["smooth"], equal_nan=True))})

    # configs[4]: long carried stream -- 10 minutes per track in 60 calls against ONE oracle run
    a = ou.synth_tracks(2, (1 if q else 10) * 60 * 48000 // H * H, sr)
    add("c5", f"configs[4] stream length: {a.shape[0]} tracks x {a.shape[1] / sr / 60:g} min ({a.shape[1] // H} frames/track) in 60 carried calls, N=2048 H=1024",
        engine_carried(a, N, H, sr, 60), ora.analyse(a, window=N, hop=H, sample_rate=sr))

    # row f4: the legacy offline analyser (AudioAnalysis.h member functions), its own comparison rule (tests/test_legacy.py)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_legacy as tl

    N, sr = 2048, 48000.0
    a = ou.make_tracks(4 if q else 24, int(sr * (2.0 if q else 8.0)), sr)
    F = 90 if q else 375
    g, la_g = fxb200.legacy_analyse(a, F, N, sr)
    pv, la_p = ou.legacy_analyse(ou.PORT_SO, a, F, N, sr)
    if os.path.exists(ou.REF_SO):
        ov, la_o = ou.legacy_analyse(ou.REF_SO, a, F, N, sr)
        assert np.array_equal(ov[..., :11], pv[..., :11], equal_nan=True)
    else:
        ov, la_o = pv, la_p
    res = tl.compare_legacy(g, la_g, ov, la_o, pv[..., ou.L["margin"]])
    res["what"] = f"legacy offline analyser: {a.shape[0]} tracks x {a.shape[1] / sr:g} s, N=2048, {F} frames per track, values from oracle/_ref, margins from the port"
    fin = np.isfinite(g[..., :10]) & np.isfinite(ov[..., :10])
    res["max_abs_err"] = {n: float(np.abs(np.where(fin[..., i], g[..., i].astype(np.float64) - ov[..., i], 0.0)).max()) for n, i in list(ou.L.items())[:10]}
    report["legacy_f4"] = res
    print("legacy_f4", {k: v for k, v in res.items() if k != "max_abs_err"}, flush=True)

    tot = {k: sum(c[k] for c in report["configs"].values()) for k in ("frames", "raw_mismatch_total", "raw_mismatch_exempt", "bad_raw", "lag_mismatch", "bad_lag", "bad_smooth", "gpu_only_low_margin_frames")}
    tot["exempt_by_cause"] = {c: sum(v["exempt_by_cause"][c] for v in report["configs"].values()) for c in ou.CAUSES}
    tot["max_abs_err"] = {n: max(v["max_abs_err"][n] for v in report["configs"].values()) for n in ou.F}
    report["totals"] = tot
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(report, open(args.out, "w"), indent=1)
    print("totals", {k: v for k, v in tot.items() if k != "max_abs_err"})
    ok = tot["bad_raw"] == 0 and tot["bad_lag"] == 0 and tot["bad_smooth"] == 0 and res["bad_continuous"] == 0 and res["bad_harmonic"] == 0
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()

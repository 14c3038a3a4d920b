#!/usr/bin/env python
"""bench.py -- analysed frames/sec of the per-frame analysis hot path on N B200s (one process per GPU).

Headline workload (BASELINE.json configs[2], the one the metric's >= 1e6 frames/s/GPU target is quoted on): 4096 tracks per
GPU, 4096-point frames, hop 1024, 48 kHz, 10 s of synthetic sine + noise per track (468 frames/track, 1.92 M
frames and 7.9 GB of fp32 audio per GPU per step -- far larger than L2, so no L2 flush is needed between steps).
A "step" analyses the next 10 s of every track: K1 k_analyse (framing, FFTs, all features) + K2 flux fix-up
+ K3 smoothing/onset, all 12 features for every frame.  Tracks shard by range across GPUs with no collective
(weak scaling: 4096 tracks per GPU); torch.distributed is used only for the barrier and the max-over-ranks time.

  value  device-resident throughput (inputs already in HBM), CUDA events on the launching stream, max over ranks
  e2e    the same metric through the C-ABI call with HOST buffers (fx_analyse_host: pinned host audio in, smoothed
         features back out, copies inside the timed region), per-step spread reported
  e2e_pcm16  the same step from 16-bit PCM host buffers (fx_analyse_host_pcm, SURVEY.md 8f3 file ingest): the samples
         cross the link at file width and are converted on the GPU (exactly, as JUCE's readers convert them)
  h2d_probe     plain pinned -> device cudaMemcpyAsync on every rank at once: the box's concurrent upload ceiling, next to
                the upload rate the e2e legs reached
  roofline      the binding roofline per BASELINE.json north_star: algorithmic FLOPs/frame (SURVEY.md 8d:
                10 N log2 N + 48 N) x frames / live-measured k_analyse time vs an FP32 FMA microbenchmark on this GPU
  roofline_hbm  algorithmic bytes/frame (4 H + 40) x frames / the same time vs MEASURED_PEAKS.json hbm_gbs
  c5            BASELINE configs[4]: 65 536 tracks x 10 min, 2048-pt frames, hop 1024, STRONG-scaled over the ranks by
                contiguous track range (fxb200.shard_tracks); slabs synthesised on the device with a continuous sample origin,
                state carried from slab to slab
  realtime      BASELINE configs[3] (N = 1 only): 512 live tracks, 256-sample blocks paced at 48 kHz for 60 s through the
                pinned ring and the engine's worker threads (tools/rt_latency.cpp): block-to-features p50 / p99 / max,
                audio-thread time per block, overruns
  cpu_baseline  the reference's own analysis classes (oracle/_ref, compiled headless) on this box's host cores,
                bounded samples of the same workload: all cores, one thread, and configs[0] on one thread

`--impl reference` times only that CPU path (all host threads), same metric / config / unit.
`--dump-outputs DIR` writes the raw and smoothed features of the last timed step (a seeded sample of rows when they are larger
than DUMP_MAX_ROWS) as finite DIR/*.npy, so that two builds can be compared output for output on the same inputs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

_REAL_STDOUT = None
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(ROOT, "feature-extractor_b200"), os.path.join(ROOT, "tests")]

WINDOW, HOP, SR = 4096, 1024, 48000.0
METRIC = "analysed frames/sec"
UNIT = "frames/s"
FP32_PEAK_THEORETICAL = 148 * 128 * 2 * 1.965e9 / 1e12       # SMs x lanes x FMA x max SM clock (MEASURED_PEAKS.json sm_max_mhz)
DUMP_MAX_ROWS = 1 << 18      # --dump-outputs: 2 blocks x (values + classes) x 2^18 rows x 12 fp32 + the fp64 row index = 52.4 MB


def algorithmic_bytes_per_frame(hop: int) -> float:
    return 4.0 * hop + 4.0 * 10            # SURVEY.md 8d: each input sample once + the 10-float feature vector


def algorithmic_flops_per_frame(n: int) -> float:
    return 10.0 * n * math.log2(n) + 48.0 * n   # SURVEY.md 8d: four real N-point transforms + O(N) feature work


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def config_dict(args, n_gpus):
    return {
        "workload": ("BASELINE configs[2]: 4096-track batch, 4096-pt frames, hop 1024, 48 kHz, all 12 features per frame"
                     if (WINDOW, HOP) == (4096, 1024) else f"exploration: {WINDOW}-pt frames, hop {HOP}, 48 kHz, all 12 features per frame"),
        "tracks_per_gpu": args.tracks, "tracks_total": args.tracks * n_gpus, "seconds_per_track": args.seconds,
        "window": WINDOW, "hop": HOP, "sample_rate": SR, "frames_per_track": int(SR * args.seconds) // HOP,
        "parallelism": f"track-range sharding x{n_gpus}, no collective",
        "l2": "inputs (7.9 GB/GPU/step) exceed L2; no flush needed",
        "signal": "SURVEY.md 8d generator (Philox-4x32-10 noise + sine, bursts, silences, three flatness regimes): k_synth on the GPU, "
                  "tests/oracle_util.py::synth_tracks on the CPU, bit-identical",
    }


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(args):
    """DRAM bytes per k_analyse launch from the committed ncu --set full capture (only valid for the default workload)."""
    p = os.path.join(ROOT, "profiles", "k_analyse_traffic.json")
    if args.tracks == 4096 and args.seconds == 10.0 and (WINDOW, HOP) == (4096, 1024) and os.path.exists(p):
        try:
            return float(json.load(open(p))["dram_bytes_per_launch"])
        except Exception:
            return None
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir: str, outputs: dict, seed: int = 0):
    """Write each [T, F, 12] device block of `outputs` as out_dir/<name>.npy, float32 [R, 12]: the same R (track, frame) rows of
    every block, all of them when T * F <= DUMP_MAX_ROWS, else a sample drawn with `seed`.  rows.npy (float64) holds their
    index t * F + f in ascending order.  Every file is finite: a non-finite value (flatness overflows to +inf on loud noise, as
    the reference's does) is written as 0 in <name>.npy and classified in <name>_nonfinite.npy (float32: 0 finite, 1 +inf,
    -1 -inf, 2 NaN); <name>.npy alone does not tell a 0 from an inf.  The engine carries its per-track state from step to step,
    so the last step depends on every step before it: dumps are comparable between runs with identical arguments, --warmup and
    --steps included."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    T, F, nf = next(iter(outputs.values())).shape
    n = T * F
    rows = np.arange(n) if n <= DUMP_MAX_ROWS else np.sort(np.random.default_rng(seed).choice(n, DUMP_MAX_ROWS, replace=False))
    for name, x in outputs.items():
        flat = x.reshape(n, nf)
        if len(rows) < n:
            flat = flat.index_select(0, torch.from_numpy(rows).to(x.device))
        v = flat.cpu().numpy().astype(np.float32)
        cls = np.select([np.isnan(v), np.isposinf(v), np.isneginf(v)], [2, 1, -1], 0).astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), np.where(cls == 0, v, np.float32(0)))
        np.save(os.path.join(out_dir, name + "_nonfinite.npy"), cls)
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------
def cpu_reference_rate(audio_np, threads: int, window=None, hop=None, sr=None):
    """frames/s of the CPU checker on audio_np [T, S]; prefers oracle/_ref (the reference's own classes)."""
    import oracle_util as ou

    ora = ou.fastest_oracle()
    t0 = time.perf_counter()
    r = ora.analyse(audio_np, threads=threads, window=window or WINDOW, hop=hop or HOP, sample_rate=sr or SR)
    dt = time.perf_counter() - t0
    frames = audio_np.shape[0] * r["frames"]
    return frames / dt, ora.kind, frames, dt


def cpu_baseline_block(args, sample_audio, cores):
    """cpu_baseline: all cores and one thread on samples of the bench workload, plus BASELINE configs[0] on one thread."""
    import oracle_util as ou

    rate, kind, frames, dt = cpu_reference_rate(sample_audio, cores)
    n1 = max(1, min(sample_audio.shape[0], 8))
    rate1, _, frames1, dt1 = cpu_reference_rate(sample_audio[:n1], 1)
    c1_audio = ou.synth_tracks(1, 441000 // 512 * 512, 44100.0)
    cpu_reference_rate(c1_audio[:, : 64 * 512], 1, 1024, 512, 44100.0)
    ratec1, _, framesc1, dtc1 = cpu_reference_rate(c1_audio, 1, 1024, 512, 44100.0)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"first {sample_audio.shape[0]} tracks x {args.seconds:g} s of the same synthetic workload ({frames} frames, {dt:.1f} s wall, {cores} threads over contiguous track ranges)",
            "single_thread": {"value": rate1, "unit": UNIT, "cores": 1, "sample": f"first {n1} tracks ({frames1} frames, {dt1:.1f} s)"},
            "c1_single_thread": {"value": ratec1, "unit": UNIT, "cores": 1,
                                 "sample": f"BASELINE configs[0]: 1 track, 44.1 kHz, 10 s, 1024-pt frames hop 512 ({framesc1} frames, {dtc1:.2f} s)",
                                 "realtime_factor": (framesc1 / dtc1) / (44100.0 / 512)}}


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation on this box's host cores (rank 0 only), fed the same Philox
    workload the GPU arm synthesises (first tracks of it)."""
    if rank != 0:
        return
    import oracle_util as ou

    cores = os.cpu_count() or 1
    n_tracks = max(8 * cores, 64)
    seconds = min(args.seconds, 10.0)
    S = (int(SR * seconds) // HOP) * HOP
    audio = ou.synth_tracks(n_tracks, S, SR)
    for _ in range(min(args.warmup, 1)):
        cpu_reference_rate(audio[: max(cores // 2, 1)], cores)
    kind = "port"
    t_all = time.perf_counter()
    for _ in range(args.steps):
        _, kind, frames, dt = cpu_reference_rate(audio, cores)
    total_dt = time.perf_counter() - t_all
    value = (n_tracks * (S // HOP) * args.steps) / total_dt
    sample = f"first {n_tracks} tracks x {seconds:g} s of the bench workload ({n_tracks * (S // HOP)} frames) per step, {cores} threads over contiguous track ranges"
    base = cpu_baseline_block(args, audio[: max(2 * cores, 16)], cores)
    base.update({"value": value, "sample": sample})
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 FFT / f64 reductions", "data": "synthetic", "config": config_dict(args, args.gpus),
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------
def run_c5(args, fxb200, torch, dist, rank, world, local_rank, dev, fp32_peak):
    """BASELINE configs[4], strong-scaled: every rank analyses its contiguous share of the 65 536 tracks for the whole 10
    minutes.  The 7.5 TB of fp32 audio never exist: each slab of every track is synthesised on the device (pure function of
    (seed, track, sample index): the stream is continuous across slabs), analysed with the per-track state carried, and
    overwritten by the next."""
    N, H = 2048, 1024
    first, T = fxb200.shard_tracks(args.c5_tracks, world, rank)
    total_frames_per_track = int(SR * 60.0 * args.c5_minutes) // H
    F = args.c5_slab_frames
    slabs = (total_frames_per_track + F - 1) // F
    S = F * H
    eng = fxb200.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, device=local_rank, ring_hops=0, max_frames_per_call=F)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    buf = torch.empty((T, S), dtype=torch.float32, device=dev)
    smooth = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
    acc = torch.zeros((T, 12), dtype=torch.float64, device=dev)

    def slab(k, timed):
        f = min(F, total_frames_per_track - k * F)
        eng.synth_device(buf.data_ptr(), S, f * H, first_track=first, first_sample=k * S, stream=sp)
        if timed:
            ev_a = torch.cuda.Event(enable_timing=True); ev_b = torch.cuda.Event(enable_timing=True)
            ev_a.record(stream)
        eng.analyse_device(buf.data_ptr(), S, f * H, None, smooth.data_ptr(), None, stream=sp)
        if timed:
            ev_b.record(stream)
            acc.add_(torch.nan_to_num(smooth[:, f - 1, :].double(), nan=0.0, posinf=0.0, neginf=0.0))      # depends on every slab
            return f, (ev_a, ev_b)
        return f, None

    for k in range(2):                      # warm-up (allocations, clocks), then a fresh stream state
        slab(k, False)
    eng.reset()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    eng.profile_enable(True)
    eng.profile_read()
    launches0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    frames_pt, pairs = 0, []
    for k in range(slabs):
        f, pr = slab(k, True)
        frames_pt += f
        pairs.append(pr)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms_all = e0.elapsed_time(e1)
    ms_an = sum(a.elapsed_time(b) for a, b in pairs)
    ms_k1, ms_post, ncalls = eng.profile_read()
    launches = eng.kernel_launches - launches0
    t = torch.tensor([ms_all, ms_an, ms_k1], dtype=torch.float64, device=dev)
    cs = torch.tensor([float(acc.sum().item())], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cs, op=dist.ReduceOp.SUM)
    eng.close()
    del buf, smooth, acc
    torch.cuda.empty_cache()
    frames_total = args.c5_tracks * frames_pt
    ms_all, ms_an, ms_k1 = (float(x) for x in t.tolist())
    flops = algorithmic_flops_per_frame(N) * T * frames_pt            # this rank's share (ranks differ by at most one track)
    return {
        "workload": f"BASELINE configs[4]: {args.c5_tracks} tracks x {args.c5_minutes:g} min at 48 kHz, 2048-pt frames, hop 1024 "
                    f"({frames_pt} frames/track); {slabs} slabs of {F} frames synthesised on the device at a continuous sample origin, state carried",
        "scaling": "strong", "n_gpus": world, "tracks_total": args.c5_tracks, "tracks_this_rank": T, "frames_total": frames_total,
        "value": frames_total / (ms_an * 1e-3), "unit": UNIT,
        "value_definition": "frames of all ranks / analysis time (K1 + K1b + K2 + K3 of every slab, CUDA events on the launching stream, max over ranks); "
                            "each slab is resident in HBM when its analysis starts",
        "seconds_analysis": ms_an * 1e-3, "seconds_including_synthesis": ms_all * 1e-3,
        "frames_per_s_including_synthesis": frames_total / (ms_all * 1e-3),
        "audio_bytes_equivalent": frames_total * H * 4, "gpu_launches": int(launches),
        "roofline": {"bound": "fp32", "kernel": "k_analyse<8>", "achieved": flops / (ms_k1 * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": flops / (ms_k1 * 1e-3) / 1e12 / fp32_peak if fp32_peak else None, "kernel_ms_total": ms_k1,
                     "kernel_share_of_analysis": ms_k1 / ms_an if ms_an else None},
        "checksum": float(cs.item()),
    }


def run_realtime(args):
    """BASELINE configs[3] through the C++ harness (tools/rt_latency.cpp, built into feature-extractor_b200/build/)."""
    exe = os.path.join(ROOT, "feature-extractor_b200", "build", "rt_latency")
    with tempfile.TemporaryDirectory() as tmp:
        if not os.path.exists(exe):         # the tree may be read-only: a harness build() did not leave is compiled outside it
            exe = os.path.join(tmp, "rt_latency")
            lib = os.path.join(ROOT, "feature-extractor_b200", "lib")
            subprocess.run(["g++", "-O2", "-std=c++17", os.path.join(ROOT, "tools", "rt_latency.cpp"), "-I" + os.path.join(ROOT, "include"),
                            "-L" + lib, "-lfxb200", "-lpthread", "-Wl,-rpath," + lib, "-o", exe], check=True)
        r = subprocess.run([exe, "512", "256", f"{args.rt_seconds:g}", "1", "128", "2048"], capture_output=True, text=True,
                           timeout=args.rt_seconds * 2 + 120)
    try:
        d = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception:
        return {"error": (r.stderr or r.stdout)[-400:], "rc": r.returncode}
    d["rc"] = r.returncode
    d["workload"] = "BASELINE configs[3]: 512 live tracks, 256-sample blocks paced at 48 kHz, 2048-pt frames hop 1024 (reference defaults), pinned ring -> 4 group workers"
    return d


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tracks", type=int, default=4096, help="tracks per GPU")
    ap.add_argument("--seconds", type=float, default=10.0, help="seconds of audio per track per step")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pcm", action="store_true", help="skip the 16-bit PCM end-to-end leg")
    ap.add_argument("--no-c5", action="store_true", help="skip the BASELINE configs[4] leg")
    ap.add_argument("--no-rt", action="store_true", help="skip the BASELINE configs[3] real-time leg")
    ap.add_argument("--c5-tracks", type=int, default=65536)
    ap.add_argument("--c5-minutes", type=float, default=10.0)
    ap.add_argument("--c5-slab-frames", type=int, default=125)
    ap.add_argument("--rt-seconds", type=float, default=60.0)
    ap.add_argument("--window", type=int, default=4096, help="exploration only: the headline workload is 4096 / 1024")
    ap.add_argument("--hop", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the features of the last timed step (rank 0's tracks) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global WINDOW, HOP
    WINDOW, HOP = args.window, args.hop

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: everything else a library prints there (NCCL's version banner, ...) goes to stderr
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import fxb200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the analysis path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    T = args.tracks
    S = (int(SR * args.seconds) // HOP) * HOP
    F = S // HOP
    frames_per_step = T * F

    eng = fxb200.Engine(n_tracks=T, window=WINDOW, hop=HOP, sample_rate=SR, device=local_rank, ring_hops=0)
    # a non-default stream: its handle is non-zero, so the library launches on exactly the stream the events are recorded on
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0
    audio = torch.empty((T, S), dtype=torch.float32, device=dev)
    raw = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
    smooth = torch.empty((T, F, 12), dtype=torch.float32, device=dev)
    eng.synth_device(audio.data_ptr(), S, S, first_track=rank * T, stream=sptr)
    torch.cuda.synchronize(dev)

    def step():
        eng.analyse_device(audio.data_ptr(), S, S, raw.data_ptr(), smooth.data_ptr(), None, stream=sptr)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # FP32 peak (registers-only FMA loop) for the compute roofline, measured on this GPU before the timed region
    fp32_peak = fxb200.measure_fp32_peak(local_rank)

    eng.profile_enable(True)
    eng.profile_read()
    launches0 = eng.kernel_launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    launches = eng.kernel_launches - launches0
    ms_k1, ms_post, ncalls = eng.profile_read()
    eng.profile_enable(False)
    ms_max = max_over_ranks(ms_total)
    value = frames_per_step * world * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"raw": raw, "smooth": smooth})

    # ---- the box's concurrent upload ceiling ---------------------------------------------------------------------
    h2d_probe = None
    if not args.no_e2e:
        barrier()
        gbs = fxb200.h2d_probe(local_rank, 1 << 30, 4, False)
        barrier()
        gbs_wc = fxb200.h2d_probe(local_rank, 1 << 30, 4, True)
        t = torch.zeros((world, 2), dtype=torch.float64, device=dev)
        t[rank, 0], t[rank, 1] = gbs, gbs_wc
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        per_rank = [float(x) for x in t[:, 0].tolist()]
        per_rank_wc = [float(x) for x in t[:, 1].tolist()]
        h2d_probe = {"what": f"4 x 1 GiB cudaMemcpyAsync pinned -> device on all {world} ranks at once (fx_h2d_probe, CUDA events)",
                     "gbs_per_rank": per_rank, "gbs_min": min(per_rank), "gbs_sum": sum(per_rank),
                     "write_combined_gbs_per_rank": per_rank_wc, "write_combined_gbs_min": min(per_rank_wc)}

    # ---- end to end through the C-ABI with host buffers ------------------------------------------------------
    e2e = None
    e2e_pcm = None
    if not args.no_e2e:
        h_audio = torch.empty((T, S), dtype=torch.float32, pin_memory=True)
        h_audio.copy_(audio)
        h_smooth = torch.empty((T, F, 12), dtype=torch.float32, pin_memory=True)
        torch.cuda.synchronize(dev)
        eng.analyse_host_ptr(h_audio.data_ptr(), S, S, None, h_smooth.data_ptr(), None)       # warm-up (allocates the pipeline slots)

        def timed_host_steps(call):
            """args.e2e_steps calls, each between barriers (host wall clock: the call returns when the results are in host
            memory); total = sum over steps of the slowest rank's time"""
            per_step = []
            for _ in range(args.e2e_steps):
                barrier()
                t0 = time.perf_counter()
                call()
                per_step.append(max_over_ranks(time.perf_counter() - t0))
            return per_step

        per = timed_host_steps(lambda: eng.analyse_host_ptr(h_audio.data_ptr(), S, S, None, h_smooth.data_ptr(), None))
        tot = sum(per)
        e2e = {"value": frames_per_step * world * args.e2e_steps / tot, "unit": UNIT,
               "h2d_bytes_per_step": T * S * 4 * world, "d2h_bytes_per_step": T * F * 12 * 4 * world,
               "steps": args.e2e_steps, "ms_per_step": {"min": 1e3 * min(per), "max": 1e3 * max(per), "mean": 1e3 * tot / len(per)},
               "api": "fx_analyse_host (pinned host audio in, smoothed features out)"}
        e2e["h2d_gbs"] = T * S * 4 * args.e2e_steps / tot / 1e9
        if h2d_probe:
            e2e["h2d_gbs_vs_probe"] = e2e["h2d_gbs"] / h2d_probe["gbs_min"]
        e2e["note"] = ("fp32 host samples as the reference's audio callback delivers them (AudioDataCollector.h:36): "
                       "bounded by the host->device link at 4 bytes/sample once the kernel outruns it; h2d_gbs is per rank, "
                       "h2d_gbs_vs_probe compares it with the slowest rank of the concurrent plain-copy probe")
        del h_audio
        # the same step from 16-bit PCM host buffers (file ingest, fx_analyse_host_pcm): half the bytes over the link;
        # the device-resident workload is quantised to 16 bits on the host first, outside the timed region
        if not args.no_pcm:
            h_pcm = torch.empty((T, S), dtype=torch.int16, pin_memory=True)
            h_pcm.copy_((audio.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round().to(torch.int16))
            torch.cuda.synchronize(dev)
            eng.analyse_host_pcm_ptr(h_pcm.data_ptr(), "s16le", 1, 0, S * 2, S, None, h_smooth.data_ptr(), None)
            per = timed_host_steps(lambda: eng.analyse_host_pcm_ptr(h_pcm.data_ptr(), "s16le", 1, 0, S * 2, S, None, h_smooth.data_ptr(), None))
            tot = sum(per)
            e2e_pcm = {"value": frames_per_step * world * args.e2e_steps / tot, "unit": UNIT,
                       "h2d_bytes_per_step": T * S * 2 * world, "d2h_bytes_per_step": T * F * 12 * 4 * world,
                       "steps": args.e2e_steps, "ms_per_step": {"min": 1e3 * min(per), "max": 1e3 * max(per), "mean": 1e3 * tot / len(per)},
                       "h2d_gbs": T * S * 2 * args.e2e_steps / tot / 1e9,
                       "api": "fx_analyse_host_pcm (pinned host 16-bit PCM in, k_pcm_decode on the GPU, smoothed features out)",
                       "parity": "decode oracle pinned to numpy / known answers only (JUCE's readers are not in the reference tree): parity unpinned"}
            del h_pcm
        del h_smooth

    # ---- CPU baseline sample is taken from the device workload before it is freed ---------------------------------
    cpu_sample = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        n_cpu_tracks = min(T, max(16 * cores, 64))
        cpu_sample = audio[:n_cpu_tracks].cpu().numpy()

    eng.close()
    del audio, raw, smooth
    torch.cuda.empty_cache()

    # ---- BASELINE configs[4], strong-scaled ------------------------------------------------------------------------
    c5 = None
    if not args.no_c5:
        barrier()
        c5 = run_c5(args, fxb200, torch, dist, rank, world, local_rank, dev, fp32_peak)
        torch.cuda.set_stream(stream)

    # ---- BASELINE configs[3] and the CPU baseline: rank 0, N = 1 only ---------------------------------------------------
    realtime = None
    cpu = None
    if rank == 0 and world == 1:
        if not args.no_rt:
            realtime = run_realtime(args)
        if cpu_sample is not None:
            import oracle_util as ou

            # the CPU generator must reproduce the device workload bit for bit (SURVEY.md 8d)
            same = bool(np.array_equal(ou.synth_tracks(2, cpu_sample.shape[1], SR), cpu_sample[:2]))
            cpu = cpu_baseline_block(args, cpu_sample, os.cpu_count() or 1)
            cpu["workload_bit_identical_to_cpu_generator"] = same

    if rank == 0:
        hbm_peak, hbm_src = measured_peaks()
        traffic = measured_traffic(args)
        k1_s = (ms_k1 * 1e-3) / max(ncalls, 1)                       # average k_analyse launch duration, CUDA events on its stream
        flops = algorithmic_flops_per_frame(WINDOW) * frames_per_step
        byts = algorithmic_bytes_per_frame(HOP) * frames_per_step
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 FFT / f64 reductions", "data": "synthetic", "config": config_dict(args, world),
            "dtype_note": "every sum is fp64 per thread (as the reference accumulates) and across the warps; across the 32 lanes of a warp the partials, "
                          "fp32-accurate squares of an fp32 spectrum, are added in fp32 (max abs error of the parity report 3.7e-5 at a 1e-4 tolerance)",
            "e2e": e2e, "e2e_pcm16": e2e_pcm, "h2d_probe": h2d_probe, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "fp32", "kernel": f"k_analyse<{WINDOW // 256}>", "achieved": flops / k1_s / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": flops / k1_s / 1e12 / fp32_peak if fp32_peak else None, "traffic": traffic,
                         "peak_source": "FMA microbenchmark on this GPU (fx_measure_fp32_peak), measured",
                         "peak_theoretical": FP32_PEAK_THEORETICAL, "frac_of_theoretical": flops / k1_s / 1e12 / FP32_PEAK_THEORETICAL,
                         "note": "binding roofline per north_star: min (HBM_BW / B, FP32_peak / F) is the FP32 term for this path",
                         "kernel_ms": k1_s * 1e3, "kernel_share_of_step": ms_k1 / ms_total if ms_total else None},
            "roofline_hbm": {"bound": "hbm", "kernel": f"k_analyse<{WINDOW // 256}>", "achieved": byts / k1_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": byts / k1_s / 1e9 / hbm_peak, "traffic": traffic, "algorithmic_bytes": byts, "peak_source": hbm_src},
            "c5": c5, "realtime": realtime, "cpu_baseline": cpu,
        }
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

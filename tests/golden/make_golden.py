"""Generate the golden fixtures in this directory from the REFERENCE ITSELF (oracle/_ref/libfxref.so = the headers
under /root/reference/Source compiled headless against oracle/juce_shim).  Run in the build container only:

    python tests/golden/make_golden.py                 # every fixture, from oracle/_ref
    python tests/golden/make_golden.py --from-port     # port_vs_reference/ only, from the port (see port_vs_reference)

The fixtures are small .npz files: seeded input (regenerated from oracle_util.make_signal, stored as a checksum
plus the first samples) and the reference's raw / smoothed feature rows and observable diagnostics.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_util as ou

CASES = {
    # name: (window, hop, sample_rate, n_tracks, seconds, mode, extra oracle config)
    "c1_n1024_h512_sr44100_modeA": (1024, 512, 44100.0, 1, 10.0, 0, {}),                 # BASELINE configs[0], verbatim run() bodies
    "c2_n2048_h512_sr48000": (2048, 512, 48000.0, 8, 2.0, 1, {}),                         # configs[1] shape, 8-track slice
    "c3_n4096_h1024_sr48000": (4096, 1024, 48000.0, 8, 2.0, 1, {}),                       # configs[2] shape, 8-track slice
    "c5_n2048_h1024_sr48000_modeA": (2048, 1024, 48000.0, 8, 3.0, 0, {}),                 # configs[3]/[4] shape (reference defaults)
    "params_n2048_h1024": (2048, 1024, 48000.0, 4, 3.0, 1, dict(gain=0.7, onset_type=2, onset_hist=7, onset_multiplier=1.2, rms_pushes=1)),
}


def main():
    ref = ou.reference()
    if ref is None:
        raise SystemExit("oracle/_ref/libfxref.so missing: run `make -C oracle` where /root/reference exists")
    for name, (N, H, sr, T, sec, mode, extra) in CASES.items():
        S = (int(sr * sec) // H) * H
        audio = ou.make_tracks(T, S, sr)
        r = ref.analyse(audio, window=N, hop=H, sample_rate=sr, mode=mode, **extra)
        np.savez_compressed(
            os.path.join(HERE, name + ".npz"),
            window=N, hop=H, sample_rate=sr, n_tracks=T, n_samples=S, mode=mode,
            extra=np.array(sorted(extra.items()), dtype=object) if extra else np.array([], dtype=object),
            audio_head=audio[:, :64], audio_sum=audio.astype(np.float64).sum(axis=1),
            raw=r["raw"], smooth=r["smooth"], lag=r["diag"][..., ou.D["lag"]], true_oer=r["diag"][..., ou.D["true_oer"]],
        )
        print(name, r["raw"].shape)


def legacy():
    """the legacy offline analyser (AudioAnalysis.h AudioAnalyser) driven headless: tests/test_legacy.py"""
    if not os.path.exists(ou.REF_SO):
        raise SystemExit("oracle/_ref/libfxref.so missing")
    N, sr, T, F, first = 2048, 48000.0, 6, 150, 2
    S = int(sr * 4.0)
    audio = ou.make_tracks(T, S, sr, first_track=first)
    out, la = ou.legacy_analyse(ou.REF_SO, audio, F, N, sr)
    np.savez_compressed(os.path.join(HERE, "legacy_n2048_sr48000.npz"), window=N, sample_rate=sr, n_tracks=T, n_samples=S, n_frames=F,
                        first_track=first, audio_head=audio[:, :64], out=out, log_attack=la)
    print("legacy", out.shape)


def port_vs_reference(from_port: bool = False):
    """port_vs_reference/: what test_port_equals_reference_on_fresh_seeds (tests/test_oracle.py) and
    test_port_is_bit_identical_to_the_reference_functions (tests/test_legacy.py) compare the port with, on their own inputs.
    Written from oracle/_ref.  With --from-port, for a tree where oracle/_ref cannot be built, the port's outputs are written
    instead and 'source' says so: the port was compared bit for bit with oracle/_ref on these inputs while the reference was
    available, and both tests check the record against oracle/_ref wherever it is built."""
    from test_legacy import CASES as LEGACY_CASES, signal
    from test_oracle import FRESH_SEED_CASES, fresh_seed_audio

    ora = ou.port() if from_port else ou.reference()
    if ora is None:
        raise SystemExit("oracle/_ref/libfxref.so missing (--from-port records the port's outputs instead)")
    lib = ou.PORT_SO if from_port else ou.REF_SO
    out_dir = os.path.join(HERE, "port_vs_reference")
    os.makedirs(out_dir, exist_ok=True)
    d = {"source": np.array(ora.kind)}
    for i, (N, H, sr) in enumerate(FRESH_SEED_CASES):
        audio = fresh_seed_audio(N, H, sr)
        r = ora.analyse(audio, window=N, hop=H, sample_rate=sr)
        d.update({f"c{i}_audio_sum": audio.astype(np.float64).sum(axis=1), f"c{i}_raw": r["raw"], f"c{i}_smooth": r["smooth"],
                  f"c{i}_lag": r["diag"][..., ou.D["lag"]]})
    np.savez_compressed(os.path.join(out_dir, "fresh_seeds.npz"), **d)
    d = {"source": np.array(ora.kind)}
    for i, (N, sr, sec, F, track) in enumerate(LEGACY_CASES):
        out, la = ou.legacy_analyse(lib, signal(N, sr, sec, track), F, N, sr)
        d.update({f"c{i}_out": out[..., :11], f"c{i}_log_attack": la})
    np.savez_compressed(os.path.join(out_dir, "legacy_cases.npz"), **d)
    print("port_vs_reference from", ora.kind)


if __name__ == "__main__":
    if "--from-port" in sys.argv:
        port_vs_reference(from_port=True)
    else:
        main()
        legacy()
        port_vs_reference()

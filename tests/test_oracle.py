"""CPU tests of the checkers under oracle/: the C restatement against (a) the golden fixtures generated from the
reference itself, (b) the headless reference build when it is present, (c) analytic known answers derived from
the reference source (SURVEY.md section 4)."""
import glob
import os

import numpy as np
import pytest

import oracle_util as ou

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = sorted(p for p in glob.glob(os.path.join(HERE, "golden", "*.npz")) if not os.path.basename(p).startswith("legacy_"))


@pytest.fixture(scope="module")
def port():
    ou.build_oracle()
    return ou.port()


def load_case(path):
    z = np.load(path, allow_pickle=True)
    N, H, sr, T, S, mode = int(z["window"]), int(z["hop"]), float(z["sample_rate"]), int(z["n_tracks"]), int(z["n_samples"]), int(z["mode"])
    extra = {k: (float(v) if isinstance(v, float) else v) for k, v in z["extra"].tolist()} if z["extra"].size else {}
    audio = ou.make_tracks(T, S, sr)
    # the generator must reproduce the exact input the fixture was made from
    assert np.array_equal(audio[:, :64], z["audio_head"])
    assert np.array_equal(audio.astype(np.float64).sum(axis=1), z["audio_sum"])
    return z, audio, dict(window=N, hop=H, sample_rate=sr, mode=mode, **extra)


def test_golden_fixtures_exist():
    assert len(GOLDEN) >= 5


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_port_matches_golden_bit_for_bit(port, path):
    z, audio, cfg = load_case(path)
    r = port.analyse(audio, **cfg)
    assert np.array_equal(r["raw"], z["raw"], equal_nan=True)
    assert np.array_equal(r["smooth"], z["smooth"], equal_nan=True)
    assert np.array_equal(r["diag"][..., ou.D["lag"]], z["lag"])
    if cfg["mode"] == 1:
        assert np.array_equal(r["diag"][..., ou.D["true_oer"]], z["true_oer"])


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_reference_build_matches_golden(path):
    ref = ou.reference()
    if ref is None:
        pytest.skip("oracle/_ref not built (no /root/reference here)")
    z, audio, cfg = load_case(path)
    r = ref.analyse(audio, **cfg)
    assert np.array_equal(r["raw"], z["raw"], equal_nan=True)
    assert np.array_equal(r["smooth"], z["smooth"], equal_nan=True)


def test_mode_a_equals_mode_b_at_half_window_hop(port):
    """Re-sequenced per-frame calls (mode B) == verbatim collector/overlapper/run() bodies (mode A) at hop N/2."""
    ref = ou.reference()
    audio = ou.make_tracks(3, 48000 * 2, 48000.0)
    for orc in [o for o in (ref, port) if o is not None]:
        a = orc.analyse(audio, window=2048, hop=1024, sample_rate=48000.0, mode=0)
        b = orc.analyse(audio, window=2048, hop=1024, sample_rate=48000.0, mode=1)
        assert np.array_equal(a["raw"], b["raw"], equal_nan=True)
        assert np.array_equal(a["smooth"], b["smooth"], equal_nan=True)


FRESH_SEED_CASES = ((1024, 256, 44100.0), (2048, 1024, 48000.0), (4096, 2048, 96000.0))
FRESH_SEED_RECORD = os.path.join(HERE, "golden", "port_vs_reference", "fresh_seeds.npz")


def fresh_seed_audio(N, H, sr):
    return ou.make_tracks(8, (int(sr * 1.5) // H) * H, sr, first_track=100, seed=7)


def test_port_equals_reference_on_fresh_seeds(port):
    """Against oracle/_ref where it is built (which must also reproduce the stored record), else against the stored record of
    this comparison (tests/golden/port_vs_reference; its 'source' says which checker wrote it, see make_golden.py)."""
    ref = ou.reference()
    rec = np.load(FRESH_SEED_RECORD)
    for i, (N, H, sr) in enumerate(FRESH_SEED_CASES):
        audio = fresh_seed_audio(N, H, sr)
        assert np.array_equal(audio.astype(np.float64).sum(axis=1), rec[f"c{i}_audio_sum"])
        stored = (rec[f"c{i}_raw"], rec[f"c{i}_smooth"], rec[f"c{i}_lag"])
        if ref is not None:
            a = ref.analyse(audio, window=N, hop=H, sample_rate=sr)
            want = (a["raw"], a["smooth"], a["diag"][..., ou.D["lag"]])
            for w, s in zip(want, stored):
                assert np.array_equal(w, s, equal_nan=True), "the stored record disagrees with oracle/_ref: regenerate it"
        else:
            want = stored
        b = port.analyse(audio, window=N, hop=H, sample_rate=sr)
        for g, w in zip((b["raw"], b["smooth"], b["diag"][..., ou.D["lag"]]), want):
            assert np.array_equal(g, w, equal_nan=True)


# ---- analytic known answers (SURVEY.md section 4) ----------------------------------------------------------
def test_kat_silence(port):
    for sr in (48000.0, 44100.0):
        r = port.analyse(np.zeros((1, 16 * 1024), np.float32), window=2048, hop=1024, sample_rate=sr)
        raw = r["raw"][0]
        expect = np.zeros(12, np.float32)
        expect[ou.F["f0"]] = np.float32(sr / 2 / 5000.0)          # lag 2: PitchAnalyser.h:146-154,176
        assert np.array_equal(raw[5], expect)
        assert (r["diag"][0, :, ou.D["lag"]] == 2).all()
        assert (r["diag"][0, :, ou.D["flat_state"]] == 3).all()


def test_kat_window_shape_and_re_squared(port):
    """FFT of an impulse at n0 has Re X[k] = w[n0] cos (2 pi k n0 / N): checks the asymmetric Bartlett window
    (RealTimeAudioAnalysis.h:148-149) through the forward FFT the reference uses."""
    N = 1024
    for n0, w in ((0, 0.0), (1, 2.0 / N), (N // 2, 1.0), (N - 1, 2.0 / N), (N // 2 + 1, 1.0 - 2.0 / N)):
        x = np.zeros(N, np.float32)
        x[n0] = 1.0
        buf = port.fft_forward(x)
        k = np.arange(N)
        assert np.allclose(buf[0::2], np.cos(2 * np.pi * k * n0 / N), atol=2e-6)
        assert np.allclose(buf[1::2], -np.sin(2 * np.pi * k * n0 / N), atol=2e-6)
    # cos at an exact bin: Re X[k0] = A N / 2; sin: Re X[k0] ~ 0 ("magnitude" is Re^2, HarmonicCharacteristics.h:63-64)
    n = np.arange(N)
    c = port.fft_forward((0.5 * np.cos(2 * np.pi * 37 * n / N)).astype(np.float32))
    s = port.fft_forward((0.5 * np.sin(2 * np.pi * 37 * n / N)).astype(np.float32))
    assert abs(c[2 * 37] - 0.25 * N) < 1e-2 and abs(s[2 * 37]) < 1e-2


def test_kat_fft_roundtrip_and_inverse_layout(port):
    rng = np.random.default_rng(3)
    N = 2048
    x = rng.standard_normal(N).astype(np.float32)
    fwd = port.fft_forward(x)
    X = np.fft.fft(x.astype(np.float64))
    assert np.allclose(fwd[0::2], X.real, atol=2e-3) and np.allclose(fwd[1::2], X.imag, atol=2e-3)
    inv = port.fft_inverse(fwd)                 # d[i] = Re / N, d[i + N] = Im / N
    assert np.allclose(inv[:N], x, atol=1e-5) and np.allclose(inv[N:], 0.0, atol=1e-5)
    # PitchAnalyser feeds Re^2 with zero imaginary parts: the imaginary output of lag 0 is exactly 0, so cnd[N] == 0
    p = np.zeros(2 * N, np.float32)
    p[0::2] = fwd[0::2] ** 2
    d = port.fft_inverse(p)
    assert d[N] == 0.0


def test_kat_first_frame_is_zero_padded(port):
    """Frame 0 = [zeros (N - H), x[0:H]] (RealTimeAudioAnalysis.h:202,214-218): RMS of frame 0 follows from it."""
    N, H = 2048, 1024
    x = np.full(4 * H, 0.25, np.float32)
    r = port.analyse(x[None, :], window=N, hop=H, sample_rate=48000.0)
    rms0 = np.float32(np.sqrt(0.25 ** 2 * H / N))
    assert np.isclose(r["raw"][0, 0, ou.F["rms"]], np.log10(np.float32(rms0 * np.float32(9.0) + np.float32(1.0))), rtol=1e-6)
    assert np.isclose(r["raw"][0, 1, ou.F["rms"]], np.log10(0.25 * 9 + 1), rtol=1e-6)


def test_kat_onset_fires_on_amplitude_step(port):
    sr, N, H = 48000.0, 2048, 1024
    n = np.arange(40 * H)
    x = (0.002 * np.sin(2 * np.pi * 440 * n / sr)).astype(np.float32)
    x[25 * H:] *= 250.0
    r = port.analyse(x[None, :], window=N, hop=H, sample_rate=sr)
    on = np.flatnonzero(r["raw"][0, :, ou.F["onset"]] > 0)
    assert on.size >= 1 and 24 <= on[0] <= 30
    assert r["raw"][0, :20, ou.F["onset"]].sum() == 0


def test_flatness_regimes_are_exercised(port):
    """sigma 0.05 -> product underflows (flatness 0), 0.5 -> overflows (inf), 0.001 -> finite (SURVEY Q7)."""
    sr, N, H = 48000.0, 2048, 1024
    audio = ou.make_tracks(8, 20 * H, sr, silence=False, bursts=False)
    r = port.analyse(audio, window=N, hop=H, sample_rate=sr)
    st = r["diag"][:, 5:, ou.D["flat_state"]]
    assert (st[0] == 1).all() and (st[6] == 2).all() and (st[7] == 0).all()
    assert np.isinf(r["raw"][6, 5:, ou.F["flatness"]]).all()
    assert (r["raw"][0, 5:, ou.F["flatness"]] == 0).all()
    fl = r["raw"][7, 5:, ou.F["flatness"]]
    assert np.isfinite(fl).all() and (fl > 0).all()


def test_compare_helper_flags_real_differences():
    a = {"raw": np.zeros((1, 4, 12), np.float32), "smooth": np.zeros((1, 4, 12), np.float32), "diag": np.ones((1, 4, 10), np.float32)}
    b = {k: v.copy() for k, v in a.items()}
    assert ou.compare(a, b)["bad_raw"] == 0
    b["raw"][0, 2, ou.F["centroid"]] = 0.01
    res = ou.compare(a, b)
    assert res["bad_raw"] == 1
    b["diag"][0, 2, ou.D["gate_margin"]] = 1e-6          # low-margin gate exempts the frame
    assert ou.compare(a, b)["bad_raw"] == 0
    a["raw"][0, 1, ou.F["flatness"]] = np.inf
    b["raw"][0, 1, ou.F["flatness"]] = np.inf
    assert ou.compare(a, b)["raw_mismatch_total"] == 1

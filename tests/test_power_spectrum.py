"""CPU tests of the power-spectrum checkers (tests/power_oracle.py: the checkers under oracle/ with fx_config.spectrum =
FX_SPECTRUM_POWER's substitution): every forward transform hands its consumers (|X[k]|, 0) instead of (Re X[k], Im X[k]), so
the features see |X|^2 per bin.
(a) a steady tone gives the same harmonic features, slope and lag at every phase (and does not in the Re^2 mode);
(b) an independent float64 restatement of RMS, centroid, spread, low-energy ratio and flux from the substituted spectra;
(c) the silence known answer; (d) the port against the reference's own classes (oracle/_ref) where that is built."""
import numpy as np
import pytest

import oracle_util as ou
import power_oracle
from f64_features import bartlett_f32

SR, N, H = 48000.0, 2048, 1024


@pytest.fixture(scope="module")
def port():
    """the power-mode port"""
    return power_oracle.port()


@pytest.fixture(scope="module")
def re_port():
    """the parity-mode port (oracle/)"""
    ou.build_oracle()
    return ou.port()


def steady_tone(phases=8, frames=24, f=1007.3, amp=0.5):
    n = np.arange(frames * H, dtype=np.float64)
    return np.stack([amp * np.sin(2 * np.pi * f * n / SR + 2 * np.pi * p / phases) for p in range(phases)]).astype(np.float32)


def test_power_mode_is_phase_invariant_on_a_steady_tone(port, re_port):
    x = steady_tone()
    spread = {}
    for mode, orc in ((0, re_port), (1, port)):
        r = orc.analyse(x, window=N, hop=H, sample_rate=SR)
        raw = r["raw"][:, 4:].astype(np.float64)            # frames 4 and later: the window is full of the tone
        spread[mode] = {k: float(raw[..., ou.F[k]].max() - raw[..., ou.F[k]].min()) for k in ("her", "inharm", "slope")}
        lags = r["diag"][:, 4:, ou.D["lag"]]
        spread[mode]["lag"] = float(lags.max() - lags.min())
        if mode == 1:
            assert np.all(raw[..., ou.F["her"]] > 0.99)       # log10 (9 HER + 1) of HER ~ 0.9994
    # power mode: the same values at every phase and frame (up to the float rounding of the transform)
    assert spread[1]["lag"] == 0.0, spread
    for k in ("her", "inharm"):
        assert spread[1][k] < 2e-5, (k, spread)
    assert spread[1]["slope"] < 2e-6, spread
    # Re^2 mode flickers over the same frames (by three orders of magnitude more): the test fails if the mode is ignored
    assert spread[0]["her"] > 0.01 and spread[0]["inharm"] > 0.01 and spread[0]["slope"] > 1e-3, spread


def test_spectral_features_match_a_float64_restatement(port, re_port):
    """RMS, centroid, spread, low-energy ratio and flux (SpectralCharacteristics.h:62-143) restated in float64 numpy on the
    port's own forward transform after the substitution X[k] -> |X[k]|, against the port's power mode."""
    x = ou.make_signal(int(1.5 * SR) // H * H, SR, track=1)         # includes a silent stretch (the previous spectrum is kept)
    r = port.analyse(x[None, :], window=N, hop=H, sample_rate=SR)["raw"][0]
    M, nyq = N // 2, SR / 2.0
    frpb = nyq / M
    fc = np.arange(M) * frpb + frpb / 2.0
    prev = np.zeros(M)
    frame = np.zeros(N, np.float32)
    checked = 0
    for f in range(len(x) // H):
        frame = np.concatenate([frame[H:], x[f * H:(f + 1) * H]])
        rms = np.float32(np.sqrt(np.sum(frame.astype(np.float64) ** 2) / N))
        log_rms = np.log10(np.float32(rms * np.float32(9.0) + np.float32(1.0)))
        assert abs(r[f, ou.F["rms"]] - log_rms) <= 1e-5
        buf = re_port.fft_forward(bartlett_f32(frame))                # the port's transform, (Re, Im) as it comes
        mag_x = np.sqrt(buf[0::2].astype(np.float64) ** 2 + buf[1::2].astype(np.float64) ** 2).astype(np.float32)
        mag = mag_x[:M].astype(np.float64) ** 2
        s = mag.sum()
        if not s > 0.05:                                              # :121-123 gated silent, previous spectrum kept
            assert r[f, ou.F["centroid"]] == 0.0 and r[f, ou.F["flux"]] == 0.0
            continue
        centroid = (fc * mag).sum() / s
        c = centroid / (nyq / 2.0)
        cn = centroid / nyq
        spread = ((fc / nyq - cn) ** 2 * mag).sum() / s / (cn * (1.0 - cn))
        ler = mag[: M // 5 + 1].sum() / s
        flux = np.clip(mag - prev, 0.0, None).sum() / (M * (M + 1) / 2.0)
        prev = mag
        want = {"centroid": np.log10(c * 9.0 + 1.0), "spread": spread, "ler": ler, "flux": flux}
        for k, v in want.items():
            assert abs(r[f, ou.F[k]] - v) <= 1e-5 * max(1.0, abs(v)), (f, k, r[f, ou.F[k]], v)
        checked += 1
    assert checked > 40


def test_kat_silence_power_mode(port):
    for sr in (48000.0, 44100.0):
        r = port.analyse(np.zeros((1, 16 * 1024), np.float32), window=2048, hop=1024, sample_rate=sr)
        expect = np.zeros(12, np.float32)
        expect[ou.F["f0"]] = np.float32(sr / 2 / 5000.0)              # lag 2: PitchAnalyser.h:146-154,176
        assert np.array_equal(r["raw"][0, 5], expect)
        assert (r["diag"][0, :, ou.D["lag"]] == 2).all()
        assert (r["diag"][0, :, ou.D["flat_state"]] == 3).all()


def test_power_mode_keeps_the_three_flatness_regimes(port):
    audio = ou.make_tracks(8, 20 * H, SR, silence=False, bursts=False)
    st = port.analyse(audio, window=N, hop=H, sample_rate=SR)["diag"][:, 5:, ou.D["flat_state"]]
    assert (st == 0).any() and (st == 1).any() and (st == 2).any()


def test_port_equals_reference_in_power_mode(port):
    """The same substitution inside the reference's unmodified classes (at the end of the shim's forward transform)."""
    ref = power_oracle.reference()
    if ref is None:
        pytest.skip("reference sources absent: the power-mode reference build cannot be made here")
    for (n, h, sr) in ((1024, 256, 44100.0), (2048, 1024, 48000.0), (4096, 2048, 96000.0)):
        audio = ou.make_tracks(6, (int(sr * 1.5) // h) * h, sr, first_track=40, seed=11)
        a = ref.analyse(audio, window=n, hop=h, sample_rate=sr)
        b = port.analyse(audio, window=n, hop=h, sample_rate=sr)
        assert np.array_equal(a["raw"], b["raw"], equal_nan=True)
        assert np.array_equal(a["smooth"], b["smooth"], equal_nan=True)
        assert np.array_equal(a["diag"][..., ou.D["lag"]], b["diag"][..., ou.D["lag"]])
    # mode A (verbatim collector / overlapper / run() bodies) = mode B at hop N/2 in this build too
    audio = ou.make_tracks(2, 24 * 1024, 48000.0)
    a = ref.analyse(audio, window=2048, hop=1024, sample_rate=48000.0, mode=0)
    b = port.analyse(audio, window=2048, hop=1024, sample_rate=48000.0, mode=0)
    assert np.array_equal(a["raw"], b["raw"], equal_nan=True)


def test_power_checker_differs_from_the_parity_checker_only_by_the_substitution(port, re_port):
    """Silence is the same in both (all spectra are 0); a signal is not; the exported transform is the port's own."""
    z = np.zeros((1, 8 * H), np.float32)
    assert np.array_equal(port.analyse(z, window=N, hop=H, sample_rate=SR)["raw"], re_port.analyse(z, window=N, hop=H, sample_rate=SR)["raw"])
    x = ou.make_tracks(1, 8 * H, SR)
    assert not np.array_equal(port.analyse(x, window=N, hop=H, sample_rate=SR)["raw"], re_port.analyse(x, window=N, hop=H, sample_rate=SR)["raw"])
    f = x[0, :N]
    assert np.array_equal(port.fft_forward(f), re_port.fft_forward(f))

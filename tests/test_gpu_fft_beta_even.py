"""At N = 4096, FFT-beta of the parity mode transforms the even part of the frame, (x[n] + x[N - n]) / 2, and computes only the
rows of the spectrum whose mirrors it does not hold; bins and lags of the skipped rows are read at N - k.  These inputs break the
mirror symmetry that the even part relies on (a frame and its mirror image differ), so a wrong mirror address or a missing row
shows up as a wrong feature or lag.  Checked against the same checkers as tests/test_gpu_parity.py at every window size (N = 2048
and 1024 run the full transform: the same cases guard that selection)."""
import numpy as np
import pytest

import oracle_util as ou

pytestmark = pytest.mark.gpu

SIZES = [(4096, 1024, 48000.0), (2048, 512, 48000.0), (1024, 256, 44100.0)]


@pytest.fixture(scope="module")
def fx():
    import fxb200

    fxb200.load_library()
    return fxb200


@pytest.fixture(scope="module")
def oracle():
    return ou.best_oracle()


def asymmetric_tracks(N, H, sr, S):
    n = np.arange(S, dtype=np.float64)
    rng = np.random.default_rng(11)
    noise = lambda a: a * rng.uniform(-1.0, 1.0, S)
    rows = []
    # impulses at window offsets n whose mirrors N - n hold nothing: one per hop, at a fixed offset inside the hop, on a weak tone
    imp = np.zeros(S)
    imp[(np.arange(S // H) * H + H // 3 + 5)] = 0.9
    rows.append(imp + 0.01 * np.sin(2 * np.pi * 440.0 * n / sr) + noise(1e-3))
    # a single impulse per window (period N) at an offset far from its mirror
    imp1 = np.zeros(S)
    imp1[np.arange(7, S, N)] = 0.8
    rows.append(imp1 + noise(2e-3))
    # a ramp with a DC offset: odd about the window centre, plus a constant
    rows.append(0.25 + 0.5 * ((n % (N + 37)) / (N + 37)) + 0.05 * np.sin(2 * np.pi * 220.0 * n / sr) + noise(1e-3))
    # a linear chirp over the whole signal: its instantaneous frequency differs between a frame and its mirror image
    f0, f1 = 80.0, 0.4 * sr / 2
    rows.append(0.5 * np.sin(2 * np.pi * (f0 * n / sr + 0.5 * (f1 - f0) * (n / sr) ** 2 / (S / sr))) + noise(1e-3))
    # a decaying tone burst that starts in the middle of a hop
    env = np.where(n % (4 * H) >= H // 2, np.exp(-((n % (4 * H)) - H // 2) / (0.7 * H)), 0.0)
    rows.append(0.6 * env * np.sin(2 * np.pi * 330.0 * n / sr + 0.4) + noise(5e-4))
    return np.stack(rows).astype(np.float32)


@pytest.mark.parametrize("N,H,sr", SIZES)
def test_asymmetric_frames_against_oracle(fx, oracle, N, H, sr):
    S = 24 * H
    audio = asymmetric_tracks(N, H, sr, S)
    o = oracle.analyse(audio, window=N, hop=H, sample_rate=sr)
    with fx.Engine(n_tracks=audio.shape[0], window=N, hop=H, sample_rate=sr) as e:
        g = e.analyse_host(audio)
    res = ou.compare(g, o)
    print(f"N={N}", ou.summary(res))
    assert res["bad_raw"] == 0, res
    assert res["bad_lag"] == 0, res
    assert res.get("bad_smooth", 0) == 0, res
    # impulses and chirps make some decisions low-margin; they are counted, never silent misses
    assert res["raw_mismatch_exempt"] <= max(2, res["frames"] // 4), res


@pytest.mark.parametrize("N,H,sr", SIZES)
def test_lags_in_every_row(fx, oracle, N, H, sr):
    """Tones whose pitch lags fall in every row of the spectrum (lag mod R1 takes every value, own rows and mirrored rows
    alike) give the oracle's lag exactly."""
    R1 = N // 256
    S = 12 * H
    n = np.arange(S, dtype=np.float64)
    rng = np.random.default_rng(5)
    # a sine of period 4 L is analysed with lag L; pick lags 16 q + r for every residue r mod R1
    lags = [16 * (2 + r) + r for r in range(R1)]
    lags = [l for l in lags if 4 * l < N]
    rows = [0.5 * np.sin(2 * np.pi * n / (4.0 * l) + 0.2 * l) + 1e-3 * rng.uniform(-1, 1, S) for l in lags]
    audio = np.stack(rows).astype(np.float32)
    o = oracle.analyse(audio, window=N, hop=H, sample_rate=sr)
    with fx.Engine(n_tracks=len(lags), window=N, hop=H, sample_rate=sr) as e:
        g = e.analyse_host(audio)
    res = ou.compare(g, o)
    print(f"N={N}", ou.summary(res))
    assert res["bad_raw"] == 0 and res["bad_lag"] == 0 and res.get("bad_smooth", 0) == 0, res
    glag = g["diag"][..., ou.D["lag"]].astype(np.int64)
    assert len({int(v) % R1 for v in glag[:, -1] if v > 0}) >= max(2, R1 // 2), glag[:, -1]

"""GPU tests of the power-spectrum mode (fx_config.spectrum = FX_SPECTRUM_POWER: |X[k]|^2 per bin instead of the reference's
Re(X[k])^2): the k_analyse<R1, MG, true> instantiations through every entry point, against the checkers run with the same
substitution (tests/power_oracle.py: reference values where they can be built, port margins) under the parity bar of
test_gpu_parity.py."""
import os

import numpy as np
import pytest

import oracle_util as ou
import power_oracle
from test_gpu_parity import CASES, assert_parity
from test_power_spectrum import steady_tone

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
POWER = 1


@pytest.fixture(scope="module")
def fx():
    import fxb200

    fxb200.load_library()
    assert fxb200.SPECTRUM_POWER == POWER
    return fxb200


@pytest.fixture(scope="module")
def oracle():
    return power_oracle.CheckedPowerOracle()


@pytest.mark.parametrize("N,H,sr,T,sec", CASES)
def test_power_parity_against_oracle(fx, oracle, N, H, sr, T, sec):
    S = (int(sr * sec) // H) * H
    audio = ou.make_tracks(T, S, sr)
    o = oracle.analyse(audio, window=N, hop=H, sample_rate=sr)
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        g = e.analyse_host(audio)
    res = ou.compare(g, o)
    assert_parity(res, f"power N={N} H={H} T={T} oracle={oracle.kind} exempt_by_cause={res['exempt_by_cause']}")
    # the mode is in effect: the same input in the parity mode gives other features
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr) as e:
        assert not np.array_equal(e.analyse_host(audio)["raw"], g["raw"], equal_nan=True)


def test_power_flatness_regimes(fx, oracle):
    """sigma 0.05 / 0.5 / 0.001 tracks: the flatness product underflows, overflows and stays finite in power mode as well"""
    N, H, sr = 2048, 1024, 48000.0
    audio = ou.make_tracks(8, 40 * H, sr, silence=False, bursts=False)
    o = oracle.analyse(audio, window=N, hop=H, sample_rate=sr)
    with fx.Engine(n_tracks=8, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        g = e.analyse_host(audio)
    assert_parity(ou.compare(g, o), "power flatness regimes")
    st = g["diag"][:, 5:, ou.D["flat_state"]]
    assert (st == 0).any() and (st == 1).any() and (st == 2).any()
    assert np.array_equal(st, o["diag"][:, 5:, ou.D["flat_state"]])


def test_power_edge_cases(fx, oracle):
    N, H, sr = 2048, 1024, 48000.0
    # silence: zeros except pitch = sr / 2 / 5000 (lag 2)
    with fx.Engine(n_tracks=1, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        r = e.analyse_host(np.zeros((1, 12 * H), np.float32))
    expect = np.zeros(12, np.float32)
    expect[ou.F["f0"]] = np.float32(sr / 2 / 5000.0)
    assert np.array_equal(r["raw"][0, 6], expect)
    assert (r["diag"][0, :, ou.D["lag"]] == 2).all()
    # full-scale square wave, DC, impulse train: decisions between rounding-noise values must all be flagged low-margin
    n = np.arange(40 * H)
    hard = np.stack([np.sign(np.sin(2 * np.pi * 1000 * n / sr)), np.ones_like(n, dtype=np.float64), (n % 997 == 0).astype(np.float64)]).astype(np.float32)
    with fx.Engine(n_tracks=3, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        g = e.analyse_host(hard)
    o = power_oracle.port().analyse(hard, window=N, hop=H, sample_rate=sr)
    assert_parity(ou.compare(g, o), "power square/dc/impulses", max_exempt_frac=1.0)
    robust = [ou.F[k] for k in ("rms", "centroid", "spread", "flatness", "ler", "flux", "slope")]
    assert ou.close(g["raw"][..., robust], o["raw"][..., robust]).all()
    # a NaN sample: lag -1 on its frames, the other tracks untouched
    x = ou.make_tracks(3, 12 * H, sr)
    x[1, 5 * H + 10] = np.nan
    o = oracle.analyse(x, window=N, hop=H, sample_rate=sr)
    with fx.Engine(n_tracks=3, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        g = e.analyse_host(x)
    assert_parity(ou.compare(g, o), "power NaN sample")
    assert (g["diag"][1, 5:7, ou.D["lag"]] == -1).all() and (o["diag"][1, 5:7, ou.D["lag"]] == -1).all()
    assert np.array_equal(np.isnan(g["raw"]), np.isnan(o["raw"]))


@pytest.mark.parametrize("N,H,sr", [(4096, 1024, 48000.0), (2048, 512, 48000.0), (1024, 512, 44100.0)])
def test_power_features_do_not_depend_on_the_diagnostics(fx, N, H, sr):
    T = 12
    audio = ou.make_tracks(T, 40 * H, sr)
    audio[3, 7 * H + 5] = np.nan
    audio[4] = 0.0
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=0, spectrum=POWER) as e:
        a = e.analyse_host(audio, want_diag=True)
        e.reset()
        b = e.analyse_host(audio, want_diag=False)
    assert np.array_equal(a["raw"], b["raw"], equal_nan=True)
    assert np.array_equal(a["smooth"], b["smooth"], equal_nan=True)


def test_power_chunked_streamed_split_and_realtime_are_bit_identical(fx):
    """K2 re-sums a chunk's first flux from the |X| spectra K1 stores: chunk and call boundaries must not show."""
    N, H, sr, T = 2048, 512, 48000.0, 3
    S = 400 * H
    audio = ou.make_tracks(T, S, sr)
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        one = e.analyse_host(audio)
        e.reset()
        cuts = [0, 7 * H, 8 * H, 150 * H, 151 * H, 333 * H, S]
        parts = [e.analyse_host(audio[:, a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(one["raw"], np.concatenate([p["raw"] for p in parts], axis=1), equal_nan=True)
    assert np.array_equal(one["smooth"], np.concatenate([p["smooth"] for p in parts], axis=1), equal_nan=True)
    with fx.Engine(n_tracks=1, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:          # one track: many chunks per track
        alone = e.analyse_host(audio[1:2])
    assert np.array_equal(alone["raw"], one["raw"][1:2], equal_nan=True)
    # real-time path: fx_push_block + fx_process reproduce the batch rows
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, ring_hops=16, tracks_per_group=2, spectrum=POWER) as e:
        done = 0
        for b0 in range(0, 120 * H, 256):
            e.push_block(audio[:, b0:b0 + 256])
            new = e.process()
            if new:
                done += new
                for t in range(T):
                    vec, idx = e.poll(t)
                    assert idx == done and np.array_equal(vec, one["smooth"][t, done - 1], equal_nan=True), (t, done)
        assert done == 120


def test_power_device_and_pcm_apis_match_host_api(fx):
    import torch

    N, H, sr, T = 4096, 1024, 48000.0, 5
    S = 60 * H
    audio = ou.make_tracks(T, S, sr)
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        host = e.analyse_host(audio)
        e.reset()
        d_audio = torch.from_numpy(audio).cuda()
        d_raw = torch.empty((T, 60, 12), device="cuda")
        d_smooth = torch.empty((T, 60, 12), device="cuda")
        d_diag = torch.empty((T, 60, 10), device="cuda")
        s = torch.cuda.current_stream()
        assert e.analyse_device(d_audio.data_ptr(), S, S, d_raw.data_ptr(), d_smooth.data_ptr(), d_diag.data_ptr(), stream=s.cuda_stream) == 60
        torch.cuda.synchronize()
        assert np.array_equal(host["raw"], d_raw.cpu().numpy(), equal_nan=True)
        assert np.array_equal(host["smooth"], d_smooth.cpu().numpy(), equal_nan=True)
        assert np.array_equal(host["diag"], d_diag.cpu().numpy(), equal_nan=True)
    # 16-bit PCM: the decoded samples are exact, so the PCM route equals the fp32 route on the decoded input
    pcm = ou.pcm_encode(np.clip(audio, -1.0, 0.999), "s16le")
    dec = np.stack([ou.pcm_decode(pcm[t], "s16le") for t in range(T)])
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=sr, spectrum=POWER) as e:
        a = e.analyse_host_pcm(pcm, "s16le")
        e.reset()
        b = e.analyse_host(dec)
    assert np.array_equal(a["raw"], b["raw"], equal_nan=True) and np.array_equal(a["smooth"], b["smooth"], equal_nan=True)


def test_power_phase_invariance_on_the_gpu(fx):
    """The CPU suite's steady tone (test_power_spectrum.py) on the GPU: the same harmonic features, slope and lag at every phase."""
    x = steady_tone()
    with fx.Engine(n_tracks=x.shape[0], window=2048, hop=1024, sample_rate=48000.0, spectrum=POWER) as e:
        g = e.analyse_host(x)
    raw = g["raw"][:, 4:].astype(np.float64)
    lags = g["diag"][:, 4:, ou.D["lag"]]
    assert lags.min() == lags.max()
    for k in ("her", "inharm"):
        assert np.ptp(raw[..., ou.F[k]]) < 2e-5, (k, np.ptp(raw[..., ou.F[k]]))
    assert np.ptp(raw[..., ou.F["slope"]]) < 2e-6


def test_engine_rejects_unknown_spectrum_mode(fx):
    with pytest.raises(fx.FxError) as ei:
        fx.Engine(n_tracks=1, spectrum=2)
    assert "(-1)" in str(ei.value) and "spectrum" in str(ei.value)
    assert fx.default_config().spectrum == 0


def test_cpp_facade_power_mode_matches_port(fx, tmp_path):
    """AudioDeviceManager constructed with FX_SPECTRUM_POWER (the facade's trailing constructor argument): the smoothed
    features of the reference wiring (256-sample device blocks, hop N/2) equal the port's power mode."""
    import subprocess

    root = os.path.dirname(HERE)
    exe = tmp_path / "facade_power_driver"
    subprocess.run(["g++", "-std=c++17", "-O2", "-o", str(exe), os.path.join(HERE, "cpp", "facade_power_driver.cpp"),
                    "-L" + os.path.join(root, "feature-extractor_b200", "lib"), "-lfxb200",
                    "-Wl,-rpath," + os.path.join(root, "feature-extractor_b200", "lib")], check=True)
    T, N, H, sr, block = 3, 2048, 1024, 48000.0, 256
    S = 60 * H
    audio = ou.make_tracks(T, S, sr)
    (tmp_path / "audio.f32").write_bytes(audio.tobytes())
    out = subprocess.run([str(exe), str(tmp_path / "audio.f32"), str(T), str(S), str(block), str(sr), str(tmp_path / "out.f32")],
                         check=True, capture_output=True, text=True).stdout
    assert "hops 60" in out
    rows = np.frombuffer((tmp_path / "out.f32").read_bytes(), np.float32).reshape(-1, T, 12)
    o = power_oracle.port().analyse(audio, window=N, hop=H, sample_rate=sr, mode=0)
    ok = ou.close(rows.transpose(1, 0, 2), o["smooth"])
    assert ok.mean() > 0.999, ok.mean()

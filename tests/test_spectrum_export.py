"""The checker of the spectrum export (tests/f64_spectrum.py), pinned without a GPU.

(a) its float64 rows agree with the port's own fp32 transform within its noise model, at every window size and in both
modes; (b) centroid, spread, low-energy ratio and flux recomputed from its rows are restate_track's values, so the rows
are the spectrum the features are defined on; (c) the library exports fx_analyse_device_spectrum and rejects a NULL
engine."""
import ctypes

import numpy as np
import pytest

import f64_features as ff
import f64_spectrum as fs
import oracle_util as ou

SR = 48000.0
SIZES = [(1024, 256), (2048, 512), (4096, 1024)]


def signals(N, H):
    """a few rows of each family (tones, noise, near-gate, full-scale, make_tracks with its silences and bursts)"""
    out = []
    for name, a in ff.families(N, H, SR, frames=N // H + 6):
        out.append((name, a[:: max(1, a.shape[0] // 3)]))
    return out


@pytest.mark.parametrize("power", [False, True], ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_rows_agree_with_the_port_transform(power, N, H):
    worst = 0.0
    for name, audio in signals(N, H):
        for row in audio:
            X64 = fs.transform(row, N, H)
            Xp = fs.transform(row, N, H, port_transform=True)
            got = fs.rows_of(Xp, power).astype(np.float32)           # the port's value, rounded once to fp32
            mag, sigma = fs.rows_of(X64, power), fs.sigma_of(X64)
            ex = fs.row_excess(got, mag, sigma)
            assert (ex <= 0.0).all(), (name, N, power, float(ex.max()), np.argwhere(ex > 0.0)[:5])
            live = sigma > 0.0
            if live.any():
                d = np.abs(np.sqrt(got.astype(np.float64)) - np.sqrt(mag))[live] / sigma[live, None]
                worst = max(worst, float(d.max()))
            zero = mag.sum(axis=1) == 0.0
            assert (got[zero] == 0.0).all(), name
    print(f"N={N} power={power}: largest |sqrt (port) - |v|| in units of sigma: {worst:.2f}")


@pytest.mark.parametrize("power", [False, True], ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_features_from_rows_are_the_restated_features(power, N, H):
    for name, audio in signals(N, H):
        for row in audio:
            mag, _ = fs.restate_rows(row, N, H, power)
            got = fs.features_from_rows(mag, SR)
            ref = ff.restate_track(row, np.full(len(row) // H, -1.0), N, H, SR, power=power)      # no lag: the harmonic body is gated
            for k in ("centroid", "spread", "ler", "flux"):
                np.testing.assert_allclose(got[k], ref[k], rtol=1e-12, atol=0.0, err_msg=f"{name} {k}")


def test_flux_reads_the_last_non_silent_row():
    """a silent row between two frames leaves the previous spectrum where it was"""
    M = 8
    a = np.zeros(M); a[1] = 1.0
    b = np.zeros(M); b[1] = 3.0; b[5] = 2.0
    got = fs.features_from_rows(np.stack([a, np.zeros(M), b]), SR)["flux"]
    assert got[1] == 0.0
    assert got[2] == ((3.0 - 1.0) + 2.0) / (M * (M + 1) / 2.0)


def test_symbol_exported_and_null_engine_rejected():
    import fxb200

    lib = fxb200.load_library()
    assert hasattr(lib, "fx_analyse_device_spectrum")
    assert "fx_analyse_device_spectrum" in fxb200.EXPORTS
    nf = ctypes.c_long(-1)
    st = lib.fx_analyse_device_spectrum(None, None, 0, 0, None, None, None, None, None, ctypes.byref(nf))
    assert st == -1                                             # FX_ERR_INVALID_ARG

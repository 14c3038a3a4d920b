"""The rows of fx_analyse_device_spectrum restated in float64, for tests only.

Row (t, f) of the exported spectrum holds, per bin m < M = N / 2, the mag[m] that the spectral body of frame f reads
(SpectralCharacteristics.h:68-73): (Re X[m])^2 in the parity mode, |X[m]|^2 in the power mode, X the transform of the
Bartlett-windowed frame with the gain applied.  This restates it as f64_features.restate_track does for its spectral body:
frames_of -> bartlett_f32 -> np.fft in float64 -> Re^2 or |X|^2, and recomputes from such rows the four features that
read nothing else (centroid, spread, low-energy ratio, flux), in restate_track's own float64 operations.

The noise model is f64_features': an fp32 transform carries an absolute error of about 1e-6 of the rms of the frame's
transform in each bin's Re (|X|).  A row value g is held to |sqrt (g) - |v|| <= 10 sigma + 1e-6 |v|, v the float64 Re
(|X|), sigma = 1e-6 x that rms.
"""
from __future__ import annotations

import numpy as np

import f64_features as ff

NOISE = 1.0e-6          # of the frame transform's rms, per bin
SIGMAS = 10.0           # allowance in units of it
REL = 1.0e-6            # relative allowance on |v| (covers the fp32 rounding of the stored square as well)


def transform(row, window, hop, gain=1.0, port_transform=False):
    """[F, M] complex: bins 0 .. M-1 of the windowed frames of one track (np.fft in float64, or the port's fp32 transform)"""
    w = ff.bartlett_f32(ff.frames_of(row, window, hop, gain))
    X = ff._port_fft(w) if port_transform else np.fft.rfft(w.astype(np.float64), axis=1)
    return X[:, : window // 2]


def rows_of(X, power):
    """float64 mag rows of a transform: Re^2 or |X|^2"""
    return (X.real ** 2 + X.imag ** 2) if power else X.real ** 2


def sigma_of(X):
    """[F] absolute per-bin noise of an fp32 transform: NOISE x the rms of the frame's transform (|X|^2 over bins 0 .. M-1)"""
    return NOISE * np.sqrt((np.abs(X) ** 2).sum(axis=1) / X.shape[1])


def restate_rows(row, window, hop, power=False, gain=1.0):
    """([F, M] float64 rows, [F] sigma) of one track"""
    X = transform(row, window, hop, gain)
    return rows_of(X, power), sigma_of(X)


def row_excess(got, mag, sigma):
    """per bin, |sqrt (got) - |v|| - (SIGMAS sigma + REL |v|), v = sqrt (mag): <= 0 passes"""
    v = np.sqrt(mag)
    return np.abs(np.sqrt(np.asarray(got, np.float64)) - v) - (SIGMAS * np.asarray(sigma)[..., None] + REL * v)


def features_from_rows(mag, sample_rate):
    """centroid, spread, ler and flux of one track's rows [F, M] (output transforms applied, 0 on silent frames), with
    restate_track's float64 operations; flux is taken against the last non-silent row (the carried previous spectrum)"""
    mag = np.asarray(mag, np.float64)
    Fn, M = mag.shape
    nyq = sample_rate / 2.0
    frpb = nyq / M
    mag_sum = mag.sum(axis=1)
    silent = ~(mag_sum > 0.05)
    safe = np.where(silent, 1.0, mag_sum)
    x = (np.arange(M) * frpb + frpb / 2.0) / nyq
    cn = (mag * x).sum(axis=1) / safe
    with np.errstate(invalid="ignore", divide="ignore"):
        out = {"centroid": np.log10((cn * 2.0) * 9.0 + 1.0),
               "spread": (((x[None, :] - cn[:, None]) ** 2) * mag).sum(axis=1) / safe / (cn * (1.0 - cn)),
               "ler": mag[:, : M // 5 + 1].sum(axis=1) / safe}
    flux = np.zeros(Fn)
    prev = np.zeros(M)
    for f in range(Fn):
        if silent[f]:
            continue
        flux[f] = np.clip(mag[f] - prev, 0.0, None).sum() / (M * (M + 1) / 2.0)
        prev = mag[f]
    out["flux"] = flux
    return {k: np.where(silent, 0.0, v) for k, v in out.items()}

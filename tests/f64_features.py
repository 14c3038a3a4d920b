"""A float64 restatement of the raw feature vector, for tests only.

The CPU port (oracle/fx_oracle.c) computes each feature in the reference's own formulation over an fp32 transform.  This
module restates the same formulas per frame in float64 numpy over np.fft, so that an implementation can be held to the
accuracy of the reference's formulation rather than to the absolute parity bar of oracle_util.compare.  An implementation
may rewrite a formula (the GPU forms spread from raw moments, for instance), but it is judged against the value of the
reference's form.

What is restated, per frame of one track (mode B framing: frames overlap by the hop, the gain multiplies the samples):
  RMS                       log10 (9 rms + 1)                                          (RealTimeAnalyser.h:207-208)
  spectral body             Bartlett window as the port applies it, np.fft of the fp32 windowed frame; per bin
                            Re^2 (parity mode) or |X|^2 (power mode); centroid, spread in the reference's own form
                            sum (x - c)^2 mag, flatness (the gated product in the log domain, with its flat-state
                            class), low-energy ratio, flux against the last non-silent frame's spectrum, silence
                            gates                                                      (SpectralCharacteristics.h:62-143)
  slope                     with the getMagnitude quirk: the largest of |raw interleaved float| over the first M
                            floats and of the per-bin magnitudes                      (:145-200)
  harmonic body             on the un-windowed frame's spectrum; HER (written to both HER and OER slots), the true
                            OER and inharmonicity, with the pitch lag taken from the checker's diagnostics
                            (HarmonicCharacteristics.h:46-259, RealTimeAnalyser.h:171)
The output transforms (log10 (9 v + 1) and so on) are applied, so values compare directly with the `raw` rows.

Slope's numerator sum (i - 1/2) e_i cancels in the reference's own form, so its rounding is relative to the scale
sum |i - 1/2| e_i (times the same factor), which restate() returns per frame as `slope_scale`.
"""
from __future__ import annotations

import numpy as np

import oracle_util as ou

FEATURES = ("rms", "f0", "centroid", "spread", "flatness", "ler", "flux", "slope", "her", "oer", "inharm", "true_oer")
LOG_DBL_MIN = np.log(2.0 ** -1022)          # below: the port's running product is subnormal and loses bits
LOG_UNDERFLOW = -1075.0 * np.log(2.0)      # below: it has rounded to zero
LOG_OVERFLOW = np.log(np.finfo(np.float64).max)


def bartlett_f32(x):
    """RealTimeWindower::scaleBufferWithBartlettWindowing as the port applies it (gain accumulated in fp32), on the last axis"""
    n = x.shape[-1]
    half = n // 2
    w = np.empty(n, np.float32)
    g, inc = np.float32(0.0), np.float32(1.0) / np.float32(half)
    for i in range(half):
        w[i] = g
        g = np.float32(g + inc)
    g, inc = np.float32(1.0), np.float32(-1.0) / np.float32(half)
    for i in range(half):
        w[half + i] = g
        g = np.float32(g + inc)
    return (x * w).astype(np.float32)


def frames_of(row, window, hop, gain=1.0):
    """[F, N] fp32 frames of one track as the overlapper builds them: zeros before the stream, samples times the gain"""
    x = (np.asarray(row, np.float32) * np.float32(gain)).astype(np.float32)
    n_frames = len(x) // hop
    padded = np.concatenate([np.zeros(window - hop, np.float32), x[: n_frames * hop]])
    idx = np.arange(n_frames)[:, None] * hop + np.arange(window)[None, :]
    return padded[idx]


def _neighbourhood_max(normed):
    """HarmonicCharacteristics.h:200-210 for every centre bin c: max of normed[c] and normed[max (c-2, 0) : min (c+2, M)]"""
    M = normed.shape[-1]
    out = normed.copy()
    for d in (-2, -1, 1):
        sh = np.full_like(normed, -np.inf)
        if d < 0:
            sh[:, -d:] = normed[:, : M + d]
        else:
            sh[:, : M - d] = normed[:, d:]
        out = np.maximum(out, sh)
    return out


def _peaks(mag):
    """binIsPeak (HarmonicCharacteristics.h:115-145) for every bin: above the mean and no larger neighbour among bin - 2,
    bin - 1 and (for bin <= M - 3) bin + 1"""
    M = mag.shape[-1]
    mean = mag.sum(axis=1, keepdims=True) / M
    peak = mag > mean
    for d in (-2, -1, 1):
        nb = np.zeros_like(peak)
        if d < 0:
            nb[:, -d:] = mag[:, : M + d] > mag[:, -d:]
        else:
            nb[:, : M - 2] = mag[:, 1: M - 1] > mag[:, : M - 2]
        peak &= ~nb
    return peak


def restate_track(row, lag, window, hop, sample_rate, power=False, gain=1.0, port_transform=False):
    """float64 features of one track.  row [S] fp32, lag [F] (the checker's diagnostics).  Returns a dict of [F] arrays:
    one per name in FEATURES, 'slope_scale', 'flat_state' (0 finite product, 1 zero, 2 inf, 3 silent frame) and
    'flat_subnormal' (the port's running product passed through the subnormal range: its bits are not comparable).
    port_transform: the same formulas over the port's fp32 transform (the reference's JUCE FFT, restated) instead of np.fft
    in float64 (test_f64_features.py checks the transform-noise model unc_* against it)."""
    fft = _port_fft if port_transform else (lambda a: np.fft.rfft(a.astype(np.float64), axis=1))
    N, H, M = window, hop, window // 2
    nyq = sample_rate / 2.0
    frpb = nyq / M
    fr = frames_of(row, N, H, gain)
    Fn = fr.shape[0]
    fr64 = fr.astype(np.float64)
    out = {}

    rms = np.sqrt((fr64 ** 2).sum(axis=1) / N)
    log_r = np.log10(rms * 9.0 + 1.0)
    out["rms"] = log_r

    # ---- spectral body ----
    X = fft(bartlett_f32(fr))[:, :M]
    mag = (X.real ** 2 + X.imag ** 2) if power else X.real ** 2
    mag_sum = mag.sum(axis=1)
    silent = ~(mag_sum > 0.05)
    safe = np.where(silent, 1.0, mag_sum)
    x = (np.arange(M) * frpb + frpb / 2.0) / nyq                       # fc / nyquist
    cn = (mag * x).sum(axis=1) / safe
    centroid = np.log10((cn * 2.0) * 9.0 + 1.0)                       # c = centroid / (nyquist / 2)
    var = (((x[None, :] - cn[:, None]) ** 2) * mag).sum(axis=1)       # the reference's own form (:135-139)
    spread = var / safe / (cn * (1.0 - cn))
    ler = mag[:, : M // 5 + 1].sum(axis=1) / safe
    eps = 0.01 * log_r
    gated = mag > eps[:, None]
    count = gated.sum(axis=1)
    flat_sum = np.where(gated, mag, 0.0).sum(axis=1)
    with np.errstate(divide="ignore"):
        cum = np.cumsum(np.where(gated, np.log(np.where(gated, mag, 1.0)), 0.0), axis=1)
    first_under = np.where((cum < LOG_UNDERFLOW).any(axis=1), np.argmax(cum < LOG_UNDERFLOW, axis=1), M)
    first_over = np.where((cum > LOG_OVERFLOW).any(axis=1), np.argmax(cum > LOG_OVERFLOW, axis=1), M)
    state = np.where(first_under < first_over, 1, np.where(first_over < first_under, 2, 0))
    cnt = np.maximum(count, 1)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        geo = np.exp(cum[:, -1] / cnt)
        flat = np.where(state == 1, 0.0, np.where(state == 2, np.inf, geo / (flat_sum / cnt)))
        flat = np.where(flat_sum > eps, flat, 0.0)
        flatness = np.log10(flat * 9.0 + 1.0)
    lowest = cum.min(axis=1, initial=0.0)
    out["flat_subnormal"] = (state != 2) & (lowest < LOG_DBL_MIN) & (lowest > LOG_UNDERFLOW - 2.0) & ~silent
    flux = np.zeros(Fn)
    prev = np.zeros(M)
    energy = (np.abs(X) ** 2).sum(axis=1)                              # |X|^2 of every bin: what the transform's rounding scales with
    prevs = np.zeros((Fn, M))                                          # the spectrum each frame's flux is measured against ...
    prev_energy = np.zeros(Fn)                                         # ... and its frame's transform energy
    prev_e = 0.0
    for f in range(Fn):
        prevs[f], prev_energy[f] = prev, prev_e
        if silent[f]:
            continue
        flux[f] = np.clip(mag[f] - prev, 0.0, None).sum() / (M * (M + 1) / 2.0)
        prev, prev_e = mag[f], energy[f]
    for k, v in (("centroid", centroid), ("spread", spread), ("flatness", flatness), ("ler", ler), ("flux", flux)):
        out[k] = np.where(silent, 0.0, v)
    out["flat_state"] = np.where(silent, 3, state)

    # slope (:145-200), the getMagnitude quirk: max |float| over the first M interleaved (Re, Im) floats = bins < M / 2
    lo = X[:, : M // 2]
    mx = np.abs(lo).max(axis=1) if power else np.maximum(np.abs(lo.real), np.abs(lo.imag)).max(axis=1)
    max_mag = np.maximum(mx, mag.max(axis=1))
    live = max_mag > 0.0001
    e = mag / np.where(live, max_mag, 1.0)[:, None]
    i = np.arange(M, dtype=np.float64)
    mean_e = e.sum(axis=1) / M
    bin_var = ((i / M - 0.5) ** 2).sum() / M
    energy_std = np.sqrt(((e - mean_e[:, None]) ** 2).sum(axis=1) / M)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = ((e * i).sum(axis=1) - M * mean_e * 0.5) / (M - 1.0) * energy_std * np.sqrt(bin_var)
        slope = r * (np.sqrt(bin_var) / energy_std)
    out["slope"] = np.where(live, slope, 0.0)
    out["slope_scale"] = np.where(live, (np.abs(i - 0.5) * e).sum(axis=1) * bin_var / (M - 1.0), 0.0)

    # ---- transform noise of each value, from the frame's own spectrum (rel_errors() allows ten times it) ----
    # Every bin's |Re| (|X|) carries the absolute rounding noise of an fp32 transform, e = 1e-6 of the rms of the frame's
    # transform (the noise model of the port's margins, taken over |X|^2: a transform rounds in proportion to the norm of its
    # input, even where Re is small), plus the fp32 rounding of the value itself (2^-23 of it: the spectrum is a float array
    # in the reference), independently per bin: dm_k = 2 sqrt (m_k) e_k + e_k^2.  A feature v moves by sum_k (dv / dm_k) dm_k;
    # its noise is the root sum of squares of those terms, after the output transform.
    ln10 = np.log(10.0)
    e_s = 1.0e-6 * np.sqrt(energy / M)[:, None] + 2.0 ** -23 * np.sqrt(mag)
    dm = 2.0 * np.sqrt(mag) * e_s + e_s ** 2
    rss = lambda g: np.sqrt(((g * dm) ** 2).sum(axis=1))
    S0, c, s = safe[:, None], cn[:, None], spread[:, None]
    D = c * (1.0 - c)
    dx = x[None, :] - c
    with np.errstate(invalid="ignore", divide="ignore"):
        unc = {"centroid": 18.0 / ((18.0 * cn + 1.0) * ln10) * rss(dx / S0),
               "spread": rss(dx ** 2 / (S0 * D) - s / S0 - s * (1.0 - 2.0 * c) / D * dx / S0),
               "ler": rss(((np.arange(M) <= M // 5)[None, :] - ler[:, None]) / S0)}
        g_flat = np.where(gated, 1.0 / (cnt[:, None] * np.where(gated, mag, 1.0)), 0.0) - np.where(gated, 1.0, 0.0) / np.where(
            flat_sum > 0, flat_sum, 1.0)[:, None]
        finite = (state == 0) & (flat_sum > eps) & (flat > 0)
        unc["flatness"] = np.where(finite, 9.0 * flat / ((9.0 * flat + 1.0) * ln10) * rss(g_flat), 0.0)
        # flux: the previous spectrum carries the same noise; bins whose increase is within the noise may flip in or out
        e_p = 1.0e-6 * np.sqrt(prev_energy / M)[:, None] + 2.0 ** -23 * np.sqrt(prevs)
        dp = 2.0 * np.sqrt(prevs) * e_p + e_p ** 2
        active = mag + dm > prevs - dp
        unc["flux"] = np.sqrt(np.where(active, dm ** 2 + dp ** 2, 0.0).sum(axis=1)) / (M * (M + 1) / 2.0)
        # slope: the bins' energies, and max_mag -- a bin's magnitude or, by the getMagnitude quirk, a raw float
        d_max = np.where(mx >= mag.max(axis=1), 1.0e-6 * np.sqrt(energy / M) + 2.0 ** -23 * mx, dm[np.arange(Fn), mag.argmax(axis=1)])
        g_slope = (i - 0.5)[None, :] * (bin_var / (M - 1.0)) / np.where(live, max_mag, 1.0)[:, None]
        unc["slope"] = np.sqrt(rss(g_slope) ** 2 + (slope / max_mag * d_max) ** 2)
    for k in ("centroid", "spread", "ler", "flatness", "flux"):
        out["unc_" + k] = np.where(silent, 0.0, np.nan_to_num(unc[k], nan=np.inf))
    out["unc_slope"] = np.where(live, np.nan_to_num(unc["slope"], nan=np.inf), 0.0)

    # ---- harmonic body: the raw, un-windowed frame (RealTimeAnalyser.h:161) ----
    lag = np.asarray(lag, np.float32)
    f0 = (nyq * 2.0) / lag.astype(np.float64)                          # PitchAnalyser.h:57
    out["f0"] = f0 / 5000.0
    R = fft(fr)[:, :M]
    hm = (R.real ** 2 + R.imag ** 2) if power else R.real ** 2
    hsum = hm.sum(axis=1)
    hmax = hm.max(axis=1)
    normed = hm / np.where(hmax > 0, hmax, 1.0)[:, None]
    nmax = _neighbourhood_max(normed)
    peaks = _peaks(hm)
    her = np.zeros(Fn)
    oer = np.zeros(Fn)
    inh = np.zeros(Fn)
    # Transform noise of the energy terms: each is the normalised magnitude of a bin whose |Re| (|X|) carries the absolute
    # rounding noise of an fp32 spectrum, e as above (1e-6 of the transform's rms plus 2^-23 of the value), i.e.
    # (2 |Re| e + e^2) / max.  On a pure
    # tone the sub-octave and even-harmonic terms are nothing but that noise.
    u_her = np.zeros(Fn)
    u_oer = np.zeros(Fn)
    u_inh = np.zeros(Fn)
    e_abs = 1.0e-6 * np.sqrt((np.abs(R) ** 2).sum(axis=1) / M)
    def u_term(f, v):
        a = np.sqrt(v * hmax[f])
        e = e_abs[f] + 2.0 ** -23 * a
        return (2.0 * a * e + e ** 2) / hmax[f]
    for f in range(Fn):
        if hsum[f] < 0.005 or not f0[f] > 0.0:
            continue
        f0_bin = int(np.floor(f0[f] / frpb))
        score = u_score = 0.0
        for lower in range(1, 16):
            lb = int(np.floor((f0[f] / 2.0 ** lower) / frpb))
            if lb != f0_bin:
                score += nmax[f, lb]
                u_score += u_term(f, nmax[f, lb])
        even = odd = u_even = u_odd = 0.0
        for h in (1, 2, 3):
            hb = int(np.floor((f0[f] * h) / frpb))
            if hb >= M:
                break
            score += nmax[f, hb]
            u_score += u_term(f, nmax[f, hb])
            if h % 2 == 0:
                even += nmax[f, hb]
                u_even += u_term(f, nmax[f, hb])
            else:
                odd += nmax[f, hb]
                u_odd += u_term(f, nmax[f, hb])
        her[f] = min(max(score / normed[f].sum(), 0.0), 1.0)
        oer[f] = min(max(even / odd, 0.0), 1.0) if odd > 0.0 else 1.0
        u_her[f] = u_score / normed[f].sum()
        u_oer[f] = (u_even + oer[f] * u_odd) / odd if odd > u_odd else np.inf
        p = np.flatnonzero(peaks[f])
        p = p[p != f0_bin]
        start = np.where(p == 0, frpb * 0.5, p * frpb)
        end = (p + 1) * frpb
        r0 = np.where(start == f0[f], 1.0, np.maximum(start, f0[f]) / np.minimum(start, f0[f]))
        r1 = np.where(end == f0[f], 1.0, np.maximum(end, f0[f]) / np.minimum(end, f0[f]))
        keep = np.floor(r0) == np.floor(r1)
        ratio = np.minimum(r0, r1)[keep]
        inh[f] = ((ratio - np.floor(ratio)) * (hm[f, p[keep]] / hsum[f])).sum()
        g = np.full(M, -inh[f] / hsum[f])
        g[p[keep]] += (ratio - np.floor(ratio)) / hsum[f]
        e = e_abs[f] + 2.0 ** -23 * np.sqrt(hm[f])
        u_inh[f] = np.sqrt(((g * (2.0 * np.sqrt(hm[f]) * e + e ** 2)) ** 2).sum())
    out["her"] = np.log10(her * 9.0 + 1.0)
    out["oer"] = out["her"]                                             # RealTimeAnalyser.h:171 stores HER in the OER slot
    out["true_oer"] = np.log10(oer * 9.0 + 1.0)
    out["inharm"] = np.log10(inh * 9.0 + 1.0)
    gate = (hsum < 0.005) | ~(f0 > 0.0)
    # the same noise after log10 (9 v + 1), for rel_errors(); 0 where the body is gated
    out["unc_her"] = np.where(gate, 0.0, 9.0 * u_her / ((9.0 * her + 1.0) * np.log(10.0)))
    out["unc_true_oer"] = np.where(gate, 0.0, 9.0 * u_oer / ((9.0 * oer + 1.0) * np.log(10.0)))
    out["unc_inharm"] = np.where(gate, 0.0, 9.0 * u_inh / ((9.0 * inh + 1.0) * np.log(10.0)))
    for k in ("her", "oer", "true_oer", "inharm"):
        out[k] = np.where(gate, 0.0, out[k])
    return out


def _port_fft(frames):
    """[F, N] fp32 -> [F, N/2 + 1] complex: the port's forward transform (oracle/fx_oracle.c fxo_fft_forward) of each frame"""
    orc = ou.port()
    N = frames.shape[1]
    out = np.empty((frames.shape[0], N // 2 + 1), np.complex128)
    for f in range(frames.shape[0]):
        b = orc.fft_forward(frames[f]).astype(np.float64)
        out[f] = b[0: N + 2: 2] + 1j * b[1: N + 2: 2]
    return out


def restate(audio, lag, window, hop, sample_rate, power=False, gain=1.0, port_transform=False):
    """restate_track over every row: a dict of [T, F] arrays"""
    per = [restate_track(audio[t], lag[t], window, hop, sample_rate, power, gain, port_transform) for t in range(audio.shape[0])]
    return {k: np.stack([p[k] for p in per]) for k in per[0]}


def values(res):
    """the compared values of a checker or GPU result (raw rows + the true OER diagnostic) as a dict of [T, F] arrays"""
    v = {k: res["raw"][..., ou.F[k]].astype(np.float64) for k in FEATURES if k != "true_oer"}
    v["true_oer"] = res["diag"][..., ou.D["true_oer"]].astype(np.float64)
    return v


def excluded(port_diag, ref, margin_tol=ou.MARGIN_TOL):
    """per feature, the [T, F] mask of values whose decisions the port itself takes with a margin below margin_tol:
    the gate margin for everything, the pitch margin for f0 / HER / OER / inharmonicity, the peak margin for
    inharmonicity, the flat margin for flatness.  Flux also hangs on the silence decisions since the last non-silent frame
    (they choose the previous spectrum), flatness on whether the port's running product went subnormal."""
    m = {k: port_diag[..., ou.D[k + "_margin"]] < margin_tol for k in ("gate", "pitch", "peak", "flat")}
    ex = {k: m["gate"].copy() for k in FEATURES}
    for k in ("f0", "her", "oer", "true_oer", "inharm"):
        ex[k] |= m["pitch"] | ~(port_diag[..., ou.D["lag"]] > 0)
    ex["inharm"] |= m["peak"]
    ex["flatness"] |= m["flat"] | ref["flat_subnormal"]
    silent = ref["flat_state"] == 3
    flux = ex["flux"]
    for t in range(flux.shape[0]):
        dirty = False
        for f in range(flux.shape[1]):
            dirty |= bool(m["gate"][t, f])
            if dirty:
                flux[t, f] = True
            if not silent[t, f] and not m["gate"][t, f]:
                dirty = False
    return ex


def rel_errors(vals, ref, ex, floor_factor=10.0):
    """per feature, the [T, F] error relative to the float64 value (to its scale for slope), after discounting
    floor_factor times the value's own transform noise (restate_track's unc_*; none for floor_factor 0); NaN where
    excluded.  A float64 value of exactly 0 admits only 0 (up to that noise); infinities compare by class."""
    err = {}
    for k in FEATURES:
        v, r = vals[k], ref[k]
        scale = ref["slope_scale"] if k == "slope" else np.abs(r)
        unc = ref.get("unc_" + ("her" if k == "oer" else k))
        with np.errstate(invalid="ignore", divide="ignore"):
            fl = 0.0 if unc is None or floor_factor == 0.0 else floor_factor * unc
            d = np.maximum(np.abs(v - r) - fl, 0.0)
            e = d / scale
        e = np.where(d == 0.0, 0.0, e)
        e = np.where(np.isinf(r) & (v == r), 0.0, e)
        e = np.where(np.isnan(e), np.inf, e)
        err[k] = np.where(ex[k], np.nan, e)
    return err


# ---------------------------------------------------------------------------------------------------------
def families(window, hop, sample_rate, frames=24, seed=0x5EED):
    """The signal families the precision tests run on, as (name, [T, S] fp32) pairs, S = frames * hop:
    pure tones at 12 frequencies from 0.02 to 0.97 of Nyquist, bin-centred and half-bin; a tone plus white noise at -40 and
    -80 dB; two tones; band-limited noise; a linear chirp; tones and noise within a factor of 2 of the silence gate (magnitude
    sum 0.05); a tone near full scale with a third harmonic; the make_tracks workload with its bursts and silences."""
    N, H, sr = window, hop, sample_rate
    S = frames * H
    n = np.arange(S, dtype=np.float64)
    rng = np.random.default_rng([seed, N, H])
    nyq = sr / 2.0
    out = []
    tones = []
    for frac in np.linspace(0.02, 0.97, 12):
        k = int(round(frac * N / 2))
        for off in (0.0, 0.5):
            f = (k + off) * sr / N
            tones.append(0.5 * np.sin(2 * np.pi * f * n / sr + rng.uniform(0, 2 * np.pi)))
    out.append(("tones", np.stack(tones)))
    rows = []
    for db in (-40.0, -80.0):
        for frac in (0.11, 0.63):
            a = 0.5 * 10.0 ** (db / 20.0)
            rows.append(0.5 * np.sin(2 * np.pi * frac * nyq * n / sr + 0.4) + a * rng.uniform(-1.0, 1.0, S) * np.sqrt(3.0))
    out.append(("tone_noise", np.stack(rows)))
    out.append(("two_tones", np.stack([0.3 * np.sin(2 * np.pi * 0.21 * nyq * n / sr) + 0.2 * np.sin(2 * np.pi * 0.37 * nyq * n / sr + 1.0),
                                       0.4 * np.sin(2 * np.pi * 0.05 * nyq * n / sr + 0.3) + 0.1 * np.sin(2 * np.pi * 0.88 * nyq * n / sr)])))
    rows = []
    for lo, hi in ((0.1, 0.15), (0.6, 0.9)):
        w = np.fft.rfft(rng.standard_normal(S))
        fr = np.fft.rfftfreq(S) * 2.0
        w[(fr < lo) | (fr > hi)] = 0.0
        v = np.fft.irfft(w, S)
        rows.append(0.2 * v / np.abs(v).max())
    out.append(("band_noise", np.stack(rows)))
    phase = 2 * np.pi * (0.01 * nyq * n / sr + 0.5 * (0.95 - 0.01) * nyq / (S / sr) * (n / sr) ** 2)
    out.append(("chirp", 0.4 * np.sin(phase)[None, :]))
    # magnitude sum of the Re^2 spectrum of an amplitude-a tone: about a^2 N^2 / 24 (Parseval with the window's N / 3)
    a_gate = np.sqrt(24 * 0.05) / N
    rows = [c * a_gate * np.sin(2 * np.pi * 0.3 * nyq * n / sr + 0.2) for c in (0.5, 0.8, 1.25, 2.0)]
    rows += [c * a_gate * np.sqrt(3.0) * rng.uniform(-1.0, 1.0, S) for c in (0.7, 1.4)]
    out.append(("near_gate", np.stack(rows)))
    out.append(("full_scale", np.stack([0.9 * np.sin(2 * np.pi * 0.07 * nyq * n / sr) + 0.09 * np.sin(2 * np.pi * 0.21 * nyq * n / sr + 0.5),
                                        np.clip(1.2 * np.sin(2 * np.pi * 0.013 * nyq * n / sr), -0.999, 0.999)])))
    out.append(("make_tracks", ou.make_tracks(8, S, sr)))
    return [(name, np.ascontiguousarray(a, dtype=np.float32)) for name, a in out]


def check(vals, ref, port_diag, bounds, what=""):
    """Compare `vals` (values()) with the restatement: per feature, |v - ref| - 10 x the value's transform noise <= bound x
    |ref| (x the scale for slope).  Returns (failures, summary): failures lists (feature, track, frame, value, float64 value,
    error) beyond the bound; summary has, per feature, the largest error with and without the noise allowance and the
    excluded count."""
    ex = excluded(port_diag, ref)
    err = rel_errors(vals, ref, ex)
    raw = rel_errors(vals, ref, ex, floor_factor=0.0)
    fails, summ = [], {"what": what, "values": int(ref["rms"].size), "max_err": {}, "max_raw_err": {}, "excluded": {}}
    for k in FEATURES:
        e = err[k]
        summ["excluded"][k] = int(ex[k].sum())
        summ["max_err"][k] = float(np.nanmax(e)) if (~np.isnan(e)).any() else 0.0
        summ["max_raw_err"][k] = float(np.nanmax(raw[k])) if (~np.isnan(raw[k])).any() else 0.0
        for t, f in zip(*np.nonzero(e > bounds.get(k, bounds["default"]))):
            fails.append((k, int(t), int(f), float(vals[k][t, f]), float(ref[k][t, f]), float(e[t, f])))
    return fails, summ

"""CPU tests of the float64 restatement (tests/f64_features.py) against the port, in both spectrum modes.

(a) Every feature of the port is within a relative 1e-5 of the float64 value of the reference's own formulation, after
    discounting ten times that value's own transform noise (f64_features.restate_track's unc_*, modelled from the frame's
    spectrum); slope relative to the scale of its cancelling numerator.  Frames whose decisions the port takes with a
    margin below 1e-4 are excluded and counted.  The largest port error per feature is printed with and without the noise
    allowance: the GPU tests (test_gpu_feature_precision.py) hold the kernels to the same bounds.
(a') The noise model is not loose and not short: the same float64 formulas over the reference's own fp32 transform (the
    port's) move every value by no more than its modelled noise.
(b) The scaling premise of the GPU's power-of-two metamorphic checks: the port is bit-invariant under x -> 2^j x in f0,
    centroid, spread, ler, HER, OER and inharmonicity, flux scales by exactly 4^j, and slope is not invariant."""
import numpy as np
import pytest

import f64_features as ff
import oracle_util as ou
import power_oracle

SR = 48000.0
SIZES = [(1024, 256), (2048, 512), (4096, 1024)]

# Relative bounds.  1e-5 for every feature the port meets at least ten times better.  RMS is log10f (9 rms + 1) in fp32
# in the reference (RealTimeAnalyser.h:207-208): near the silence gate the fp32 rounding of 1 + 9 rms is 2e-5 .. 6e-5 of
# the logarithm in the port, so its bound is ten times the port's worst.
BOUNDS = {"default": 1e-5, "rms": 6e-4}


def checker(power):
    return power_oracle.port() if power else ou.port()


def compare_port(power, N, H, families):
    orc = checker(power)
    fails, worst, raw, excl, total = [], {k: 0.0 for k in ff.FEATURES}, {k: 0.0 for k in ff.FEATURES}, {k: 0 for k in ff.FEATURES}, 0
    for name, audio in families:
        o = orc.analyse(audio, window=N, hop=H, sample_rate=SR)
        lag = o["diag"][..., ou.D["lag"]]
        ref = ff.restate(audio, lag, N, H, SR, power=power)
        f, s = ff.check(ff.values(o), ref, o["diag"], BOUNDS, name)
        fails += [(name,) + x for x in f]
        total += s["values"]
        for k in ff.FEATURES:
            worst[k] = max(worst[k], s["max_err"][k])
            raw[k] = max(raw[k], s["max_raw_err"][k])
            excl[k] += s["excluded"][k]
    return fails, worst, raw, excl, total


@pytest.mark.parametrize("power", [False, True], ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_port_matches_the_float64_restatement(power, N, H):
    fams = ff.families(N, H, SR, frames=N // H + 20)
    fails, worst, raw, excl, total = compare_port(power, N, H, fams)
    print(f"port vs float64, {'power' if power else 're_squared'} N={N} H={H}: {total} frames; largest relative error per feature "
          "(without / beyond ten times the value's transform noise):",
          {k: f"{raw[k]:.1e} / {worst[k]:.1e}" for k in ff.FEATURES}, "excluded", excl)
    assert not fails, fails[:20]
    # the bounds are ten times above the port's worst error beyond the transform noise (a yardstick, not a second port)
    for k, v in worst.items():
        assert v <= BOUNDS.get(k, BOUNDS["default"]) / 10.0 + 1e-12, (k, v)
    assert max(excl.values()) <= 0.05 * total, excl


@pytest.mark.parametrize("power", [False, True], ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_transform_noise_model_covers_the_reference_transform(power, N, H):
    """unc_* is a per-value model (1e-6 of the transform's rms plus the fp32 rounding of each bin, root sum of squares over
    the bins).  Over the port's fp32 transform the float64 formulas move by at most that much (observed: up to 0.96 of it),
    so the ten-fold allowance of check() is the reference's own accuracy with a margin, value by value."""
    worst = {}
    for name, audio in ff.families(N, H, SR, frames=N // H + 20):
        o = checker(power).analyse(audio, window=N, hop=H, sample_rate=SR)
        lag = o["diag"][..., ou.D["lag"]]
        ref = ff.restate(audio, lag, N, H, SR, power=power)
        ref32 = ff.restate(audio, lag, N, H, SR, power=power, port_transform=True)
        ex = ff.excluded(o["diag"], ref)
        for k in ("centroid", "spread", "ler", "flatness", "flux", "slope", "her", "true_oer", "inharm"):
            with np.errstate(invalid="ignore"):
                d = np.abs(ref32[k] - ref[k])              # inf - inf where both products overflowed (flat state 2)
            d = np.where(np.isinf(ref[k]) & (ref32[k] == ref[k]), 0.0, d)
            u = ref["unc_" + k]
            m = ~ex[k] & (d > 0)
            assert np.isfinite(d[m]).all(), (name, k)
            with np.errstate(divide="ignore"):
                worst[k] = max(worst.get(k, 0.0), float((d[m] / u[m]).max()) if m.any() else 0.0)
    print(f"largest |fp32-transform value - float64 value| / modelled noise, {'power' if power else 're_squared'} N={N}:",
          {k: f"{v:.2f}" for k, v in worst.items()})
    for k, v in worst.items():
        assert v <= 2.0, (k, v)


def test_restatement_sees_a_wrong_spread():
    """The yardstick is sharp: a spread off by 1e-4 relative on a tone is a failure, and so is one off by 3e-4 on most steady
    frames of the lowest tones (0.02 .. 0.1 of Nyquist), by 1e-2 on all of them.  (Where the hop meets the tone near a zero of
    Re, the Re^2 spectrum is small against |X| and the transform's noise allows up to 3e-3 of the spread.)"""
    N, H = 2048, 512
    audio = ff.families(N, H, SR, frames=16)[0][1][:4]
    o = ou.port().analyse(audio, window=N, hop=H, sample_rate=SR)
    lag = o["diag"][..., ou.D["lag"]]
    ref = ff.restate(audio, lag, N, H, SR)
    v = ff.values(o)
    assert not ff.check(v, ref, o["diag"], BOUNDS)[0]
    steady = {(t, f) for t in range(4) for f in range(N // H, 16)}
    for rel, share in ((1e-4, 0.3), (3e-4, 0.8), (1e-2, 1.0)):
        w = dict(v, spread=v["spread"] * (1.0 + rel))
        fails = ff.check(w, ref, o["diag"], BOUNDS)[0]
        assert {f[0] for f in fails} == {"spread"}
        caught = {(t, f) for _, t, f, *_ in fails} & steady
        assert len(caught) >= share * len(steady), (rel, len(caught), len(steady))


INVARIANT = ("f0", "centroid", "spread", "ler", "her", "oer", "inharm")


@pytest.mark.parametrize("power", [False, True], ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_port_is_bit_invariant_under_power_of_two_scaling(power, N, H):
    orc = checker(power)
    audio = ou.make_tracks(8, (N // H + 16) * H, SR, silence=False, bursts=False)
    base = orc.analyse(audio, window=N, hop=H, sample_rate=SR)
    slope_moved = False
    for j in (-4, -2, 1, 3):
        o = orc.analyse(audio * np.float32(2.0 ** j), window=N, hop=H, sample_rate=SR)
        assert np.array_equal(o["diag"][..., ou.D["lag"]], base["diag"][..., ou.D["lag"]]), j
        for k in INVARIANT:
            assert np.array_equal(o["raw"][..., ou.F[k]], base["raw"][..., ou.F[k]]), (j, k)
        assert np.array_equal(o["diag"][..., ou.D["true_oer"]], base["diag"][..., ou.D["true_oer"]]), j
        assert np.array_equal(o["raw"][..., ou.F["flux"]], base["raw"][..., ou.F["flux"]] * np.float32(4.0 ** j)), j
        slope_moved |= not np.array_equal(o["raw"][..., ou.F["slope"]], base["raw"][..., ou.F["slope"]])
    # max_mag mixes max |raw float| (linear in x) with max Re^2 (quadratic): the getMagnitude quirk breaks the invariance
    # (in the power mode the raw floats are |X|, whose largest square wins on these signals)
    assert slope_moved or power

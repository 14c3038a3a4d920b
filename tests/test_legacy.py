"""The legacy offline analyser (SURVEY.md section 8 row f4): struct AudioAnalyser of AudioAnalysis.h, whose feature block is
commented out at the reference's own call site (:219-247) while its member functions are intact.

CPU: the plain-C port (oracle/fx_oracle.c) against the reference's own member functions (oracle/_ref, where built) and against
the golden fixture generated from them.  GPU: fx_legacy_analyse_host through the C ABI against the same checker -- values from
oracle/_ref, decision margins from the port."""
import os

import numpy as np
import pytest

import oracle_util as ou

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "legacy_n2048_sr48000.npz")
CASES = [(2048, 48000.0, 2.0, 90, 3), (1024, 44100.0, 3.0, 200, 6), (4096, 48000.0, 4.0, 64, 7), (2048, 48000.0, 3.0, 1, 1), (2048, 48000.0, 5.0, 400, 1)]


def signal(N, sr, sec, track):
    return ou.make_tracks(1, int(sr * sec), sr, first_track=track)


CASES_RECORD = os.path.join(HERE, "golden", "port_vs_reference", "legacy_cases.npz")


@pytest.mark.parametrize("N,sr,sec,F,track", CASES)
def test_port_is_bit_identical_to_the_reference_functions(N, sr, sec, F, track):
    """Against oracle/_ref where it is built (which must also reproduce the stored record), else against the stored record of
    this comparison (tests/golden/port_vs_reference; its 'source' says which checker wrote it, see make_golden.py)."""
    ou.port()
    a = signal(N, sr, sec, track)
    rec = np.load(CASES_RECORD)
    key = f"c{CASES.index((N, sr, sec, F, track))}"
    rec_out, rec_la = rec[key + "_out"], rec[key + "_log_attack"]
    if os.path.exists(ou.REF_SO):
        r, lr = ou.legacy_analyse(ou.REF_SO, a, F, N, sr)
        assert (r[..., ou.L["margin"]] == -1).all()
        assert np.array_equal(r[..., :11], rec_out, equal_nan=True) and np.array_equal(lr, rec_la, equal_nan=True), \
            "the stored record disagrees with oracle/_ref: regenerate it"
    else:
        r, lr = rec_out, rec_la
    p, lp = ou.legacy_analyse(ou.PORT_SO, a, F, N, sr)
    assert np.array_equal(r[..., :11], p[..., :11], equal_nan=True)
    assert np.array_equal(lr, lp, equal_nan=True)
    assert (p[..., ou.L["margin"]] >= 0).all()


def test_port_against_golden_fixture():
    ou.port()
    z = np.load(GOLDEN)
    a = ou.make_tracks(int(z["n_tracks"]), int(z["n_samples"]), float(z["sample_rate"]), first_track=int(z["first_track"]))
    assert np.array_equal(a[:, :64], z["audio_head"])
    p, lp = ou.legacy_analyse(ou.PORT_SO, a, int(z["n_frames"]), int(z["window"]), float(z["sample_rate"]))
    assert np.array_equal(p[..., :11], z["out"][..., :11], equal_nan=True)
    assert np.array_equal(lp, z["log_attack"], equal_nan=True)
    # the fixture exercises the path: several f0 values, the previousF0 rule, overflowing and finite products, silent frames
    f0 = z["out"][..., ou.L["f0"]]
    assert len(np.unique(f0)) >= 4 and np.isinf(z["out"][..., ou.L["flatness"]]).any() and (z["out"][..., ou.L["flatness"]] == 0).any()


def compare_legacy(g, la_g, o, la_o, margin):
    """Per-frame comparison.  Continuous slots within 1e-4 (inf / NaN by class).  The harmonic slots hang on integer decisions
    (peak bins, the best interval, the previousF0 rule) and on state carried from frame to frame: a frame is exempt when the
    oracle's own margin is below 1e-4, or while the carried f0 differs because an earlier exempt frame went the other way."""
    T, F, _ = o.shape
    cont = [ou.L[k] for k in ("centroid", "spread", "flatness", "flux", "slope", "zcr", "energy")]
    harm = [ou.L[k] for k in ("f0", "her", "inharm")]
    ok_c = ou.close(g[..., cont], o[..., cont])
    ok_h = ou.close(g[..., harm], o[..., harm]) & (g[..., ou.L["num_peaks"]] == o[..., ou.L["num_peaks"]])[..., None]
    low = margin < ou.MARGIN_TOL
    exempt = np.zeros((T, F), bool)
    for t in range(T):
        diverged = False
        for f in range(F):
            exempt[t, f] = low[t, f] or diverged
            diverged = (diverged or low[t, f]) and not bool(ou.close(g[t, f, ou.L["f0"]], o[t, f, ou.L["f0"]]))
    return {"frames": T * F, "bad_continuous": int((~ok_c & ~low[..., None]).sum()), "continuous_mismatch": int((~ok_c).sum()),
            "bad_harmonic": int((~ok_h & ~exempt[..., None]).sum()), "harmonic_mismatch_frames": int((~ok_h).any(axis=-1).sum()),
            "exempt_frames": int(exempt.sum()), "low_margin_frames": int(low.sum()),
            "log_attack_equal": bool(np.array_equal(la_g, la_o, equal_nan=True))}


@pytest.mark.gpu
@pytest.mark.parametrize("N,sr,sec,F,T", [(2048, 48000.0, 4.0, 180, 12), (1024, 44100.0, 3.0, 250, 8), (4096, 48000.0, 6.0, 100, 8), (2048, 48000.0, 2.0, 1, 3)])
def test_gpu_legacy_analyser_matches_the_reference_functions(N, sr, sec, F, T):
    import fxb200

    a = ou.make_tracks(T, int(sr * sec), sr)
    g, la_g = fxb200.legacy_analyse(a, F, N, sr)
    p, la_p = ou.legacy_analyse(ou.PORT_SO, a, F, N, sr)
    if os.path.exists(ou.REF_SO):
        o, la_o = ou.legacy_analyse(ou.REF_SO, a, F, N, sr)
        assert np.array_equal(o[..., :11], p[..., :11], equal_nan=True)
    else:
        o, la_o = p, la_p
    res = compare_legacy(g, la_g, o, la_o, p[..., ou.L["margin"]])
    print(res)
    assert res["bad_continuous"] == 0 and res["bad_harmonic"] == 0, res
    # exemptions must stay the exception, and the path must have been exercised
    assert res["harmonic_mismatch_frames"] <= 0.05 * res["frames"] + 2, res
    assert (o[..., ou.L["f0"]] > 0).mean() > 0.5 and len(np.unique(o[..., ou.L["f0"]])) >= (2 if F > 1 else 1)
    # zero crossings are integer counts: exact
    assert np.array_equal(g[..., ou.L["zcr"]], o[..., ou.L["zcr"]])
    if F > 1:
        assert res["log_attack_equal"] or (p[..., ou.L["margin"]] < 1e-3).any()


@pytest.mark.gpu
def test_gpu_legacy_analyser_edge_cases():
    import fxb200

    sr, N = 48000.0, 2048
    a = np.zeros((2, 48000), np.float32)                      # silence: every gate closed
    a[1, 20000:20010] = 0.5                                    # one click: a few frames see a flat-ish spectrum
    g, la = fxb200.legacy_analyse(a, 40, N, sr)
    o, lo = ou.legacy_analyse(ou.PORT_SO, a, 40, N, sr)
    assert np.array_equal(g[0, :, :10], o[0, :, :10]) and (g[0, :, :10] == 0).all()
    res = compare_legacy(g, la, o, lo, o[..., ou.L["margin"]])
    assert res["bad_continuous"] == 0 and res["bad_harmonic"] == 0, res
    with pytest.raises(fxb200.FxError):
        fxb200.legacy_analyse(a, 40, 3000, sr)

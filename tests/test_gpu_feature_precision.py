"""GPU features against the float64 restatement of the reference's formulation (tests/f64_features.py), at relative
precision, in both spectrum modes (run with `-m gpu`).

The parity tests accept |gpu - ref| <= 1e-4 max (1, |ref|), an absolute 1e-4 for the many feature values far below 1.
Here every value is held to the relative bounds the port meets (test_f64_features.py), after discounting ten times that
value's own transform noise (modelled from the frame's spectrum, f64_features.restate_track's unc_*); decisions the port
takes with a margin below 1e-4 are excluded and counted, and no feature may have more than 5 % of its values excluded.
(a) the signal families of f64_features.families() and a shape cut into many chunks per track (K2's stitched fluxes);
(b) invariants at full size and a sample of it against the restatement; (c) power-of-two metamorphic checks: scaled input, engine gain and gain changes between calls change
nothing but what scales with the input in the reference's arithmetic, bit for bit."""
import numpy as np
import pytest

import f64_features as ff
import oracle_util as ou
import power_oracle
from test_f64_features import BOUNDS, INVARIANT

pytestmark = pytest.mark.gpu

SR = 48000.0
SIZES = [(1024, 256), (2048, 512), (4096, 1024)]
MODES = [(False, 0), (True, 1)]
# Largest share of a feature's values that the port's low-margin decisions may exclude, so that no test passes by excluding.
# Flatness gets more room: on the frames around make_tracks' silences many bins sit at the flatness gate (Re^2 vs
# 0.01 log rms), and the reference itself decides that gate within 1e-4 on 6 % of the chunked shape's frames (12 % of one
# track's).
MAX_EXCLUDED = {"default": 0.05, "flatness": 0.08}


def assert_excluded_share(counts, total, what):
    share = {k: v / total for k, v in counts.items()}
    print(what, "excluded share per feature", {k: f"{v:.3f}" for k, v in share.items() if v})
    for k, v in share.items():
        assert v <= MAX_EXCLUDED.get(k, MAX_EXCLUDED["default"]), (what, k, v)


@pytest.fixture(scope="module")
def fx():
    import fxb200

    fxb200.load_library()
    return fxb200


def port(power):
    return power_oracle.port() if power else ou.port()


def gpu_run(fx, audio, N, H, mode, **kw):
    with fx.Engine(n_tracks=audio.shape[0], window=N, hop=H, sample_rate=SR, spectrum=mode, **kw) as e:
        return e.analyse_host(np.ascontiguousarray(audio))


def against_restatement(fx, audio, N, H, power, mode, what, g=None):
    """GPU vs float64 under BOUNDS; returns (failures, summary, excluded values per feature)"""
    o = port(power).analyse(audio, window=N, hop=H, sample_rate=SR)
    if g is None:
        g = gpu_run(fx, audio, N, H, mode)
    lag = o["diag"][..., ou.D["lag"]]
    ref = ff.restate(audio, lag, N, H, SR, power=power)
    fails, summ = ff.check(ff.values(g), ref, o["diag"], BOUNDS, what)
    ex = ff.excluded(o["diag"], ref)
    # the lag is exact wherever the port's pitch and gate decisions are clear (the restatement takes it from the port)
    lag_ok = ex["f0"] | (g["diag"][..., ou.D["lag"]] == lag)
    assert lag_ok.all(), (what, np.argwhere(~lag_ok)[:10])
    return fails, summ, {k: int(v.sum()) for k, v in ex.items()}


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_gpu_matches_the_float64_restatement(fx, power, mode, N, H):
    fails, counts, total, worst, raw = [], {k: 0 for k in ff.FEATURES}, 0, {k: 0.0 for k in ff.FEATURES}, {k: 0.0 for k in ff.FEATURES}
    for name, audio in ff.families(N, H, SR, frames=N // H + 20):
        f, s, ex = against_restatement(fx, audio, N, H, power, mode, name)
        fails += [(name,) + x for x in f]
        total += s["values"]
        for k in ff.FEATURES:
            worst[k] = max(worst[k], s["max_err"][k])
            raw[k] = max(raw[k], s["max_raw_err"][k])
            counts[k] += ex[k]
    print(f"gpu vs float64, mode {mode} N={N} H={H}: largest relative error per feature (without / beyond ten times the "
          "value's transform noise):", {k: f"{raw[k]:.1e} / {worst[k]:.1e}" for k in ff.FEATURES})
    assert not fails, (len(fails), fails[:20])
    assert_excluded_share(counts, total, f"mode {mode} N={N}")


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
def test_gpu_precision_with_many_chunks_per_track(fx, power, mode):
    """3 tracks x 400 frames: many chunks per track, so K2's stitched fluxes at the chunk starts are among the values"""
    N, H = 2048, 512
    audio = ou.make_tracks(3, 400 * H, SR)
    fails, summ, ex = against_restatement(fx, audio, N, H, power, mode, "chunked")
    print("chunked", mode, summ)
    assert not fails, (len(fails), fails[:20])
    assert_excluded_share(ex, summ["values"], f"chunked, mode {mode}")


def test_full_size_invariants_and_sample(fx):
    """BASELINE configs[2] width (4096 tracks, N = 4096, H = 1024, the synth workload, 2 s): on every non-silent frame
    spread >= 0, flux >= 0 and 0 <= ler <= 1; 64 tracks of it against the restatement."""
    import torch

    N, H, T = 4096, 1024, 4096
    S = 2 * 48000 // H * H
    F = S // H
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR) as e:
        d_audio = torch.empty((T, S), device="cuda")
        e.synth_device(d_audio.data_ptr(), S, S, first_track=0)
        d_raw = torch.empty((T, F, 12), device="cuda")
        d_diag = torch.empty((T, F, 10), device="cuda")
        e.analyse_device(d_audio.data_ptr(), S, S, d_raw.data_ptr(), None, d_diag.data_ptr())
        e.flush()
        torch.cuda.synchronize()
        raw, diag = d_raw.cpu().numpy(), d_diag.cpu().numpy()
        ids = np.arange(0, T, T // 64)
        sample = d_audio[torch.from_numpy(ids).cuda()].cpu().numpy()
    live = diag[..., ou.D["flat_state"]] != 3
    assert live.mean() > 0.5
    for k, lo, hi in (("spread", 0.0, np.inf), ("flux", 0.0, np.inf), ("ler", 0.0, 1.0)):
        v = raw[..., ou.F[k]][live]
        bad = ~((v >= lo) & (v <= hi))
        assert not bad.any(), (k, int(bad.sum()), v[bad][:10])
    g = {"raw": raw[ids], "diag": diag[ids]}
    fails, summ, ex = against_restatement(fx, sample, N, H, False, 0, "full-size sample", g=g)
    print(summ)
    assert not fails, (len(fails), fails[:20])
    assert_excluded_share(ex, summ["values"], "full-size sample")


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_power_of_two_scaling_is_exact(fx, power, mode, N, H):
    """x -> 2^j x (j where the port crosses no gate, test_f64_features.py) leaves lag, f0, centroid, spread, ler, HER, OER,
    the true OER and inharmonicity bit-identical and multiplies flux by exactly 4^j.  Engine gain 2^j equals the pre-scaled
    input at gain 1 in all raw and smoothed features, and so do power-of-two gains changed between calls (the carried
    overlap is rescaled, k_tail_scale)."""
    audio = ou.make_tracks(8, (N // H + 16) * H, SR, silence=False, bursts=False)
    base = gpu_run(fx, audio, N, H, mode)
    for j in (-4, -2, 1, 3):
        s = np.float32(2.0 ** j)
        g = gpu_run(fx, audio * s, N, H, mode)
        assert np.array_equal(g["diag"][..., ou.D["lag"]], base["diag"][..., ou.D["lag"]]), j
        for k in INVARIANT:
            assert np.array_equal(g["raw"][..., ou.F[k]], base["raw"][..., ou.F[k]]), (j, k)
        assert np.array_equal(g["diag"][..., ou.D["true_oer"]], base["diag"][..., ou.D["true_oer"]]), j
        assert np.array_equal(g["raw"][..., ou.F["flux"]], base["raw"][..., ou.F["flux"]] * np.float32(4.0 ** j)), j
        gained = gpu_run(fx, audio, N, H, mode, gain=float(s))
        assert np.array_equal(gained["raw"], g["raw"], equal_nan=True), j
        assert np.array_equal(gained["smooth"], g["smooth"], equal_nan=True), j
    # gains changed between calls: the stream pre-multiplied call by call, at gain 1
    F = audio.shape[1] // H
    cuts = [(0, 5, 0.5), (5, 6, 4.0), (6, F - 4, 0.125), (F - 4, F, 2.0)]
    pre = audio.copy()
    parts = []
    with fx.Engine(n_tracks=audio.shape[0], window=N, hop=H, sample_rate=SR, spectrum=mode, ring_hops=0) as e:
        for a, b, gain in cuts:
            pre[:, a * H: b * H] *= np.float32(gain)
            e.set_gain(gain)
            parts.append(e.analyse_host(np.ascontiguousarray(audio[:, a * H: b * H])))
    got = {k: np.concatenate([p[k] for p in parts], axis=1) for k in ("raw", "smooth")}
    want = gpu_run(fx, pre, N, H, mode)
    assert np.array_equal(got["raw"], want["raw"], equal_nan=True)
    assert np.array_equal(got["smooth"], want["smooth"], equal_nan=True)

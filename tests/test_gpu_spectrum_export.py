"""fx_analyse_device_spectrum on the GPU (run with `-m gpu`): the exported rows against the float64 restatement
(tests/f64_spectrum.py), and what the export must leave alone.

1. rows match the restatement at N = 1024 / 2048 / 4096 in both modes, on the signal families of f64_features and
   make_tracks; all-zero frames give exact zeros;
2. raw, smooth and diag are bit-identical with and without the export, diagnostics on and off;
3. one call, three uneven calls and a track cut into many chunks give bit-identical rows (a silent run crosses a boundary);
4. centroid, spread, ler and flux recomputed from the rows match the GPU's own raw features;
5. an engine gain of 2^k scales every row by exactly 4^k, and so does a gain changed between calls on the frames whose
   window lies wholly after the change;
6. an output above 2^31 elements (64-bit row index), with a sentinel after its end;
7. argument handling: misaligned d_spec, d_spec = NULL, the real-time workers running."""
import ctypes

import numpy as np
import pytest

import f64_features as ff
import f64_spectrum as fs
import oracle_util as ou
import power_oracle
from test_f64_features import BOUNDS

pytestmark = pytest.mark.gpu

SR = 48000.0
SIZES = [(1024, 256), (2048, 512), (4096, 1024)]
MODES = [(False, 0), (True, 1)]
ROW_FEATURES = ("centroid", "spread", "ler", "flux")


@pytest.fixture(scope="module")
def fx():
    import fxb200

    fxb200.load_library()
    return fxb200


def run(fx, audio, N, H, mode, spec=True, diag=True, cuts=None, gains=None, **kw):
    """analyse_device over `audio` [T, S] in calls [a, b) of hops (cuts; default one call), gain gains[i] for call i;
    returns numpy raw, smooth, diag (None when off) and spec (None when off), concatenated along frames"""
    import torch

    T, S = audio.shape
    F = S // H
    cuts = cuts or [(0, F)]
    out = {k: [] for k in ("raw", "smooth", "diag", "spec")}
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, spectrum=mode, ring_hops=0, **kw) as e:
        d_audio = torch.from_numpy(np.ascontiguousarray(audio)).cuda()
        for i, (a, b) in enumerate(cuts):
            if gains is not None:
                e.set_gain(float(gains[i]))
            f = b - a
            d_raw = torch.empty((T, f, 12), device="cuda")
            d_smooth = torch.empty((T, f, 12), device="cuda")
            d_diag = torch.empty((T, f, 10), device="cuda") if diag else None
            d_spec = torch.full((T, f, N // 2), np.nan, device="cuda") if spec else None
            nf = e.analyse_device(d_audio.data_ptr() + 4 * a * H, S, f * H, d_raw.data_ptr(), d_smooth.data_ptr(),
                                  d_diag.data_ptr() if diag else None, d_spec_ptr=d_spec.data_ptr() if spec else None)
            assert nf == f
            torch.cuda.synchronize()
            out["raw"].append(d_raw.cpu().numpy())
            out["smooth"].append(d_smooth.cpu().numpy())
            out["diag"].append(d_diag.cpu().numpy() if diag else None)
            out["spec"].append(d_spec.cpu().numpy() if spec else None)
    return {k: (np.concatenate(v, axis=1) if v[0] is not None else None) for k, v in out.items()}


def signal_sets(N, H):
    """f64_features' families, and make_tracks behind a lead-in of silence long enough for all-zero frames"""
    F = N // H + 12
    late = ou.make_tracks(4, F * H, SR)
    late[:, : (N // H + 2) * H] = 0.0
    return ff.families(N, H, SR, frames=F) + [("late_start", late)]


def check_rows(spec, audio, N, H, power, what, gain=1.0):
    """every row against the restatement; all-zero frames exactly zero.  Returns the largest excess in units of sigma."""
    worst = 0.0
    for t in range(audio.shape[0]):
        mag, sigma = fs.restate_rows(audio[t], N, H, power, gain)
        got = spec[t]
        assert np.isfinite(got).all() and (got >= 0.0).all(), (what, t)
        ex = fs.row_excess(got, mag, sigma)
        assert (ex <= 0.0).all(), (what, t, float(ex.max()), np.argwhere(ex > 0.0)[:5])
        zero = mag.sum(axis=1) == 0.0
        assert (got[zero] == 0.0).all(), (what, t)
        live = sigma > 0.0
        if live.any():
            d = np.abs(np.sqrt(got.astype(np.float64)) - np.sqrt(mag))[live] / sigma[live, None]
            worst = max(worst, float(d.max()))
    return worst


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_rows_match_the_restatement_and_perturb_nothing(fx, power, mode, N, H):
    """(1) and (2): rows against float64; raw / smooth / diag bit-identical with the export off, diagnostics on and off"""
    worst, zero_frames = 0.0, 0
    for name, audio in signal_sets(N, H):
        g = run(fx, audio, N, H, mode)
        worst = max(worst, check_rows(g["spec"], audio, N, H, power, name))
        zero_frames += int((g["spec"].max(axis=2) == 0.0).sum())
        plain = run(fx, audio, N, H, mode, spec=False)
        for k in ("raw", "smooth", "diag"):
            assert np.array_equal(g[k], plain[k], equal_nan=True), (name, k)
        no_diag = run(fx, audio, N, H, mode, diag=False)
        no_diag_plain = run(fx, audio, N, H, mode, spec=False, diag=False)
        assert np.array_equal(no_diag["spec"], g["spec"]), name
        for k in ("raw", "smooth"):
            assert np.array_equal(no_diag[k], no_diag_plain[k], equal_nan=True), (name, k)
            assert np.array_equal(no_diag[k], g[k], equal_nan=True), (name, k)
    print(f"mode {mode} N={N}: largest |sqrt (row) - |v|| = {worst:.2f} sigma; {zero_frames} all-zero rows")
    assert zero_frames > 0                      # the zero-padded stream start and make_tracks' silences are covered


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_call_boundaries_do_not_matter(fx, power, mode, N, H):
    """(3) one call, three uneven calls and one track cut into many chunks (two tracks, 300 frames) give the same bits"""
    F = 300
    audio = ou.make_tracks(2, F * H, SR)
    audio[:, 97 * H: 131 * H] = 0.0                        # a silent run across the boundary at frame 120
    one = run(fx, audio, N, H, mode)
    three = run(fx, audio, N, H, mode, cuts=[(0, 120), (120, 121), (121, F)])
    assert np.array_equal(one["spec"], three["spec"])
    assert np.array_equal(one["raw"], three["raw"], equal_nan=True)
    many = run(fx, audio, N, H, mode, cuts=[(a, min(F, a + 37)) for a in range(0, F, 37)])
    assert np.array_equal(one["spec"], many["spec"])
    silent = one["spec"][:, 97 + N // H: 131].max(axis=2)
    assert (silent == 0.0).all()
    check_rows(one["spec"], audio, N, H, power, "make_tracks, 300 frames")


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_rows_match_the_gpu_features(fx, power, mode, N, H):
    """(4) centroid, spread, ler and flux from the exported rows against the GPU's raw features: relative BOUNDS after ten
    times each value's transform noise, the port's low-margin decisions excluded (test_gpu_feature_precision.py)"""
    orc = power_oracle.port() if power else ou.port()
    total, excluded, worst = 0, {k: 0 for k in ROW_FEATURES}, {k: 0.0 for k in ROW_FEATURES}
    for name, audio in signal_sets(N, H):
        g = run(fx, audio, N, H, mode)
        o = orc.analyse(audio, window=N, hop=H, sample_rate=SR)
        ref = ff.restate(audio, o["diag"][..., ou.D["lag"]], N, H, SR, power=power)
        from_rows = [fs.features_from_rows(g["spec"][t], SR) for t in range(audio.shape[0])]
        for k in ROW_FEATURES:
            ref[k] = np.stack([r[k] for r in from_rows])
        ex = ff.excluded(o["diag"], ref)
        err = ff.rel_errors(ff.values(g), ref, ex)
        total += audio.shape[0] * g["spec"].shape[1]
        for k in ROW_FEATURES:
            excluded[k] += int(ex[k].sum())
            e = err[k]
            if (~np.isnan(e)).any():
                worst[k] = max(worst[k], float(np.nanmax(e)))
            bad = np.argwhere(e > BOUNDS["default"])
            assert not len(bad), (name, k, bad[:5], [float(e[tuple(i)]) for i in bad[:5]])
    print(f"mode {mode} N={N}: largest relative error of the row features", worst, "excluded", excluded, "of", total)
    for k in ROW_FEATURES:
        assert excluded[k] <= 0.05 * total, (k, excluded[k], total)


@pytest.mark.parametrize("power,mode", MODES, ids=["re_squared", "power"])
@pytest.mark.parametrize("N,H", SIZES)
def test_power_of_two_gain_scales_rows_exactly(fx, power, mode, N, H):
    """(5) gain 2^k: every row times exactly 4^k; a gain changed between calls: the frames whose window lies wholly after
    the change, and every frame equals the stream pre-multiplied call by call"""
    F = N // H + 24
    audio = ou.make_tracks(4, F * H, SR, silence=False, bursts=False)
    base = run(fx, audio, N, H, mode)["spec"]
    for k in (-3, -1, 2):
        g = run(fx, audio, N, H, mode, gain=float(2.0 ** k))["spec"]
        assert np.array_equal(g, base * np.float32(4.0 ** k)), k
    NB = N // H
    c = 10
    for k in (-2, 1):
        got = run(fx, audio, N, H, mode, cuts=[(0, c), (c, F)], gains=[1.0, 2.0 ** k])["spec"]
        after = slice(c + NB - 1, F)                       # frame f covers hop blocks f - NB + 1 .. f
        assert np.array_equal(got[:, after], base[:, after] * np.float32(4.0 ** k)), k
        assert np.array_equal(got[:, :c], base[:, :c]), k
        pre = audio.copy()
        pre[:, c * H:] *= np.float32(2.0 ** k)
        assert np.array_equal(got, run(fx, pre, N, H, mode)["spec"]), k


def test_output_above_2_to_the_31_elements(fx):
    """(6) 4096 tracks x 300 frames at N = 4096: 2.5e9 elements (10 GB).  A sentinel after the end stays untouched; rows of
    the first and last 8 tracks match the restatement."""
    import torch

    N, H, T, F = 4096, 1024, 4096, 300
    M, S = N // 2, F * H
    n = T * F * M
    assert n > 2 ** 31
    tail = 4096
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, ring_hops=0) as e:
        d_audio = torch.empty((T, S), device="cuda")
        e.synth_device(d_audio.data_ptr(), S, S, first_track=0)
        d_spec = torch.empty(n + tail, device="cuda")
        d_spec[n:] = -7.0
        d_raw = torch.empty((T, F, 12), device="cuda")
        assert e.analyse_device(d_audio.data_ptr(), S, S, d_raw.data_ptr(), None, None, d_spec_ptr=d_spec.data_ptr()) == F
        e.flush()
        torch.cuda.synchronize()
        assert bool((d_spec[n:] == -7.0).all())
        ids = list(range(8)) + list(range(T - 8, T))
        spec = d_spec[:n].view(T, F, M)[ids].cpu().numpy()
        audio = d_audio[ids].cpu().numpy()
        del d_spec, d_audio
    frames = np.array([0, 1, 2, 3, 150, 151, 298, 299])
    for i, t in enumerate(ids):
        mag, sigma = fs.restate_rows(audio[i], N, H, False)
        ex = fs.row_excess(spec[i][frames], mag[frames], sigma[frames])
        assert (ex <= 0.0).all(), (t, float(ex.max()))


def test_argument_handling(fx):
    """(7) a misaligned d_spec is rejected and nothing is written; d_spec = NULL is fx_analyse_device; the call is refused
    while the real-time workers run"""
    import torch

    N, H, T = 1024, 256, 4
    F = 20
    audio = ou.make_tracks(T, F * H, SR)
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, ring_hops=0) as e:
        d_audio = torch.from_numpy(audio).cuda()
        d_raw = torch.zeros((T, F, 12), device="cuda")
        buf = torch.full((T * F * N // 2 + 4,), -3.0, device="cuda")
        lib, nf = e.lib, ctypes.c_long(0)
        for off in (4, 8, 12):
            st = lib.fx_analyse_device_spectrum(e._h, d_audio.data_ptr(), F * H, F * H, d_raw.data_ptr(), None, None,
                                                buf.data_ptr() + off, None, ctypes.byref(nf))
            assert st == -1, off                                 # FX_ERR_INVALID_ARG
        torch.cuda.synchronize()
        assert bool((buf == -3.0).all()) and bool((d_raw == 0.0).all())
        # nothing was analysed either: the stream still starts at sample 0
        with_spec = run(fx, audio, N, H, 0)
        ref = e.analyse_host(audio)
        assert np.array_equal(with_spec["raw"], ref["raw"], equal_nan=True)
    for mode in (0, 1):
        a = run(fx, audio, N, H, mode, spec=False)
        with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, spectrum=mode, ring_hops=0) as e:
            d_audio = torch.from_numpy(audio).cuda()
            outs = [torch.empty((T, F, w), device="cuda") for w in (12, 12, 10)]
            st = e.lib.fx_analyse_device_spectrum(e._h, d_audio.data_ptr(), F * H, F * H, *[o.data_ptr() for o in outs], None,
                                                  None, ctypes.byref(nf))
            assert st == 0 and nf.value == F
            torch.cuda.synchronize()
            for k, o in zip(("raw", "smooth", "diag"), outs):
                assert np.array_equal(o.cpu().numpy(), a[k], equal_nan=True), (mode, k)
    with fx.Engine(n_tracks=T, window=N, hop=H, sample_rate=SR, ring_hops=8) as e:
        d_audio = torch.from_numpy(audio).cuda()
        d_spec = torch.full((T, F, N // 2), -3.0, device="cuda")
        e.rt_start(lambda *a: None)
        try:
            with pytest.raises(fx.FxError):
                e.analyse_device(d_audio.data_ptr(), F * H, F * H, None, None, None, d_spec_ptr=d_spec.data_ptr())
        finally:
            e.rt_stop()
        torch.cuda.synchronize()
        assert bool((d_spec == -3.0).all())

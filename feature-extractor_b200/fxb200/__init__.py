"""fxb200 -- thin ctypes binding over the C ABI of libfxb200.so (include/fx_engine.h).

This is plumbing for tests and bench.py: the product is the shared library (CUDA kernels for sm_100a behind
a C ABI) and the C++ facade in ../host/.  There is deliberately no CPU fallback here: if the library is
missing or no CUDA device is present, construction fails loudly.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_long, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FXB200_LIB selects another build of the same library (kernel experiments); the default is the in-tree build
LIB_PATH = os.environ.get("FXB200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libfxb200.so")

NUM_FEATURES = 12
NUM_DIAG = 10
FEATURES = ("onset", "rms", "f0", "centroid", "spread", "flatness", "ler", "flux", "slope", "her", "oer", "inharm")
DIAG = ("true_oer", "lag", "pitch_margin", "num_peaks", "peak_margin", "flat_count", "flat_margin", "gate_margin",
        "onset_margin", "flat_state")
# OSCFeatureAnalysisOutput.h:107 (12 floats on the wire) and README.md:55-57 (10 floats documented)
OSC_ORDER_CODE = ("onset", "rms", "f0", "centroid", "slope", "spread", "flatness", "ler", "flux", "her", "oer", "inharm")
OSC_ORDER_README = ("onset", "rms", "f0", "centroid", "slope", "spread", "flatness", "flux", "her", "inharm")

# every symbol include/fx_engine.h declares
EXPORTS = (
    "fx_default_config", "fx_engine_create", "fx_engine_destroy", "fx_last_error", "fx_version", "fx_set_gain",
    "fx_set_onset", "fx_reset", "fx_analyse_host", "fx_analyse_device", "fx_push_block", "fx_process",
    "fx_poll_features", "fx_flush", "fx_osc_order", "fx_synth_device", "fx_kernel_launches",
    "fx_profile_enable", "fx_profile_read", "fx_measure_fp32_peak",
    "fx_pcm_bytes_per_sample", "fx_analyse_host_pcm", "fx_decode_pcm_device",
    "fx_poll_block", "fx_rt_start", "fx_rt_stop", "fx_set_features_callback", "fx_set_track_active", "fx_clear_buffer",
    "fx_set_sample_rate", "fx_rt_get_stats", "fx_osc_encode_tracks", "fx_synth_device_at", "fx_h2d_probe",
    "fx_legacy_analyse_host", "fx_analyse_device_spectrum",
)

# fx_engine.h FX_LEGACY_*: output slots of the legacy offline analyser (AudioAnalysis.h)
LEGACY = ("centroid", "spread", "flatness", "flux", "slope", "f0", "her", "inharm", "zcr", "energy", "num_peaks", "product_state")

# fx_engine.h FX_PCM_*: sample encodings of WAV (little endian) and AIFF (big endian) data chunks
PCM_FORMATS = {"u8": 1, "s8": 2, "s16le": 3, "s16be": 4, "s24le": 5, "s24be": 6, "s32le": 7, "s32be": 8, "f32le": 9, "f32be": 10}


class Config(ctypes.Structure):
    _fields_ = [
        ("n_tracks", c_int), ("window", c_int), ("hop", c_int), ("sample_rate", c_double), ("device", c_int),
        ("rms_pushes_per_frame", c_int), ("onset_type", c_int), ("onset_hist", c_int), ("onset_multiplier", c_float),
        ("gain", c_float), ("max_frames_per_call", c_long), ("ring_hops", c_int), ("tracks_per_group", c_int),
        ("spectrum", c_int),
    ]


class RtStats(ctypes.Structure):
    _fields_ = [("batches", c_uint64), ("hops", c_uint64), ("overruns", c_uint64), ("batch_ms_mean", c_double), ("batch_ms_max", c_double)]


# fx_config.spectrum (fx_engine.h FX_SPECTRUM_*): the reference's Re(X)^2 per bin (default), or |X|^2 -- Engine(spectrum=SPECTRUM_POWER)
SPECTRUM_RE_SQUARED = 0
SPECTRUM_POWER = 1

FEATURES_CALLBACK = ctypes.CFUNCTYPE(None, c_void_p, c_int, c_int, c_uint64, c_int)


class FxError(RuntimeError):
    pass


_lib = None


def load_library(path: str | None = None) -> ctypes.CDLL:
    """Load libfxb200.so and declare its prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FxError(f"{p} not found: build it with `make -C feature-extractor_b200` (or __graft_entry__.build()); "
                      "there is no CPU fallback")
    lib = ctypes.CDLL(p)
    lib.fx_default_config.argtypes = [POINTER(Config)]
    lib.fx_default_config.restype = None
    lib.fx_engine_create.argtypes = [POINTER(Config), POINTER(c_void_p)]
    lib.fx_engine_create.restype = c_int
    lib.fx_engine_destroy.argtypes = [c_void_p]
    lib.fx_engine_destroy.restype = c_int
    lib.fx_last_error.argtypes = [c_void_p]
    lib.fx_last_error.restype = c_char_p
    lib.fx_version.argtypes = []
    lib.fx_version.restype = c_char_p
    lib.fx_set_gain.argtypes = [c_void_p, c_int, c_float]
    lib.fx_set_gain.restype = c_int
    lib.fx_set_onset.argtypes = [c_void_p, c_int, c_int, c_int, c_float]
    lib.fx_set_onset.restype = c_int
    lib.fx_reset.argtypes = [c_void_p]
    lib.fx_reset.restype = c_int
    lib.fx_analyse_host.argtypes = [c_void_p, c_void_p, c_long, c_long, c_void_p, c_void_p, c_void_p, POINTER(c_long)]
    lib.fx_analyse_host.restype = c_int
    lib.fx_analyse_device.argtypes = [c_void_p, c_void_p, c_long, c_long, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_long)]
    lib.fx_analyse_device.restype = c_int
    lib.fx_analyse_device_spectrum.argtypes = [c_void_p, c_void_p, c_long, c_long, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                               POINTER(c_long)]
    lib.fx_analyse_device_spectrum.restype = c_int
    lib.fx_push_block.argtypes = [c_void_p, c_int, c_int, POINTER(c_void_p), c_int]
    lib.fx_push_block.restype = c_int
    lib.fx_process.argtypes = [c_void_p, POINTER(c_long)]
    lib.fx_process.restype = c_int
    lib.fx_poll_features.argtypes = [c_void_p, c_int, POINTER(c_float), POINTER(c_uint64)]
    lib.fx_poll_features.restype = c_int
    lib.fx_flush.argtypes = [c_void_p]
    lib.fx_flush.restype = c_int
    lib.fx_osc_order.argtypes = [POINTER(c_float), POINTER(c_float), c_int]
    lib.fx_osc_order.restype = c_int
    lib.fx_synth_device.argtypes = [c_void_p, c_void_p, c_long, c_long, c_long, c_uint64, c_void_p]
    lib.fx_synth_device.restype = c_int
    lib.fx_kernel_launches.argtypes = [c_void_p]
    lib.fx_kernel_launches.restype = c_uint64
    lib.fx_profile_enable.argtypes = [c_void_p, c_int]
    lib.fx_profile_enable.restype = c_int
    lib.fx_profile_read.argtypes = [c_void_p, POINTER(c_double), POINTER(c_double), POINTER(c_long)]
    lib.fx_profile_read.restype = c_int
    lib.fx_measure_fp32_peak.argtypes = [c_int, POINTER(c_double)]
    lib.fx_measure_fp32_peak.restype = c_int
    lib.fx_pcm_bytes_per_sample.argtypes = [c_int]
    lib.fx_pcm_bytes_per_sample.restype = c_int
    lib.fx_analyse_host_pcm.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_long, c_long, c_void_p, c_void_p, c_void_p, POINTER(c_long)]
    lib.fx_analyse_host_pcm.restype = c_int
    lib.fx_decode_pcm_device.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_long, c_long, c_long, c_void_p, c_long, c_void_p]
    lib.fx_decode_pcm_device.restype = c_int
    lib.fx_poll_block.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p]
    lib.fx_poll_block.restype = c_int
    lib.fx_rt_start.argtypes = [c_void_p]
    lib.fx_rt_start.restype = c_int
    lib.fx_rt_stop.argtypes = [c_void_p]
    lib.fx_rt_stop.restype = c_int
    lib.fx_set_features_callback.argtypes = [c_void_p, FEATURES_CALLBACK, c_void_p]
    lib.fx_set_features_callback.restype = c_int
    lib.fx_set_track_active.argtypes = [c_void_p, c_int, c_int, c_int]
    lib.fx_set_track_active.restype = c_int
    lib.fx_clear_buffer.argtypes = [c_void_p, c_int]
    lib.fx_clear_buffer.restype = c_int
    lib.fx_set_sample_rate.argtypes = [c_void_p, c_double]
    lib.fx_set_sample_rate.restype = c_int
    lib.fx_rt_get_stats.argtypes = [c_void_p, POINTER(RtStats), c_int]
    lib.fx_rt_get_stats.restype = c_int
    lib.fx_osc_encode_tracks.argtypes = [c_void_p, POINTER(c_int), c_int, POINTER(c_char_p), c_int, c_void_p, c_int, POINTER(c_int)]
    lib.fx_osc_encode_tracks.restype = c_int
    lib.fx_synth_device_at.argtypes = [c_void_p, c_void_p, c_long, c_long, c_long, c_long, c_uint64, c_void_p]
    lib.fx_synth_device_at.restype = c_int
    lib.fx_h2d_probe.argtypes = [c_int, c_long, c_int, c_int, POINTER(c_double)]
    lib.fx_h2d_probe.restype = c_int
    lib.fx_legacy_analyse_host.argtypes = [c_int, c_int, c_double, c_void_p, c_long, c_long, c_int, c_int, c_void_p, c_void_p]
    lib.fx_legacy_analyse_host.restype = c_int
    if path is None:
        _lib = lib
    return lib


def default_config(**overrides) -> Config:
    lib = load_library()
    cfg = Config()
    lib.fx_default_config(ctypes.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise TypeError(f"unknown fx_config field {k!r}")
        setattr(cfg, k, v)
    return cfg


class Engine:
    """One fx_engine: n_tracks analyser tracks on one GPU."""

    def __init__(self, **cfg):
        self.lib = load_library()
        self.cfg = default_config(**cfg)
        self._h = c_void_p()
        st = self.lib.fx_engine_create(ctypes.byref(self.cfg), ctypes.byref(self._h))
        if st != 0:
            raise FxError(f"fx_engine_create failed ({st}): {self.lib.fx_last_error(None).decode()}")

    # -- lifetime ------------------------------------------------------------------------------------------
    def close(self):
        if self._h:
            self.lib.fx_engine_destroy(self._h)
            self._h = c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st: int, what: str):
        if st != 0:
            raise FxError(f"{what} failed ({st}): {self.lib.fx_last_error(self._h).decode()}")

    # -- parameters ----------------------------------------------------------------------------------------
    def set_gain(self, gain: float, track: int = -1):
        self._check(self.lib.fx_set_gain(self._h, track, gain), "fx_set_gain")

    def set_onset(self, type: int = 1, hist_len: int = 5, multiplier: float = 1.7, track: int = -1):
        self._check(self.lib.fx_set_onset(self._h, track, type, hist_len, multiplier), "fx_set_onset")

    def reset(self):
        self._check(self.lib.fx_reset(self._h), "fx_reset")

    def set_sample_rate(self, sample_rate: float):
        self._check(self.lib.fx_set_sample_rate(self._h, sample_rate), "fx_set_sample_rate")

    def set_track_active(self, track: int, active: bool, reset_state: bool = False):
        self._check(self.lib.fx_set_track_active(self._h, track, 1 if active else 0, 1 if reset_state else 0), "fx_set_track_active")

    def clear_buffer(self, track: int = -1):
        self._check(self.lib.fx_clear_buffer(self._h, track), "fx_clear_buffer")

    # -- batch analysis, host buffers ------------------------------------------------------------------------
    def analyse_host(self, audio: np.ndarray, want_raw=True, want_smooth=True, want_diag=True):
        """audio: float32 [n_tracks, n_samples] (C-contiguous rows).  Returns dict of numpy arrays."""
        a = np.ascontiguousarray(audio, dtype=np.float32)
        if a.ndim != 2 or a.shape[0] != self.cfg.n_tracks:
            raise ValueError("audio must be [n_tracks, n_samples]")
        T, S = a.shape
        F = S // self.cfg.hop
        raw = np.empty((T, F, NUM_FEATURES), np.float32) if want_raw else None
        smooth = np.empty((T, F, NUM_FEATURES), np.float32) if want_smooth else None
        diag = np.empty((T, F, NUM_DIAG), np.float32) if want_diag else None
        nf = c_long(0)
        st = self.lib.fx_analyse_host(self._h, a.ctypes.data, S, S,
                                      raw.ctypes.data if want_raw else None,
                                      smooth.ctypes.data if want_smooth else None,
                                      diag.ctypes.data if want_diag else None, ctypes.byref(nf))
        self._check(st, "fx_analyse_host")
        assert nf.value == F
        return {"raw": raw, "smooth": smooth, "diag": diag, "frames": F}

    def analyse_host_ptr(self, audio_ptr: int, track_stride: int, n_samples: int, raw_ptr=None, smooth_ptr=None, diag_ptr=None) -> int:
        nf = c_long(0)
        st = self.lib.fx_analyse_host(self._h, audio_ptr, track_stride, n_samples, raw_ptr, smooth_ptr, diag_ptr, ctypes.byref(nf))
        self._check(st, "fx_analyse_host")
        return nf.value

    # -- file ingest: interleaved PCM rows (bytes as they lie in a WAV / AIFF data chunk) ------------------------
    def analyse_host_pcm(self, pcm: np.ndarray, fmt: str, n_channels: int = 1, channel: int = 0,
                         want_raw=True, want_smooth=True, want_diag=True):
        """pcm: uint8 [n_tracks, row_bytes]; each row holds sample frames of n_channels interleaved samples."""
        b = np.ascontiguousarray(pcm).view(np.uint8)
        if b.ndim != 2 or b.shape[0] != self.cfg.n_tracks:
            raise ValueError("pcm must be [n_tracks, row_bytes]")
        code = PCM_FORMATS[fmt]
        bps = self.lib.fx_pcm_bytes_per_sample(code)
        T, row = b.shape
        S = row // (bps * n_channels)
        F = S // self.cfg.hop
        raw = np.empty((T, F, NUM_FEATURES), np.float32) if want_raw else None
        smooth = np.empty((T, F, NUM_FEATURES), np.float32) if want_smooth else None
        diag = np.empty((T, F, NUM_DIAG), np.float32) if want_diag else None
        nf = c_long(0)
        st = self.lib.fx_analyse_host_pcm(self._h, b.ctypes.data, code, n_channels, channel, row, S,
                                          raw.ctypes.data if want_raw else None,
                                          smooth.ctypes.data if want_smooth else None,
                                          diag.ctypes.data if want_diag else None, ctypes.byref(nf))
        self._check(st, "fx_analyse_host_pcm")
        assert nf.value == F
        return {"raw": raw, "smooth": smooth, "diag": diag, "frames": F}

    def analyse_host_pcm_ptr(self, pcm_ptr: int, fmt: str, n_channels: int, channel: int, track_stride_bytes: int, n_samples: int,
                             raw_ptr=None, smooth_ptr=None, diag_ptr=None) -> int:
        nf = c_long(0)
        st = self.lib.fx_analyse_host_pcm(self._h, pcm_ptr, PCM_FORMATS[fmt], n_channels, channel, track_stride_bytes, n_samples,
                                          raw_ptr, smooth_ptr, diag_ptr, ctypes.byref(nf))
        self._check(st, "fx_analyse_host_pcm")
        return nf.value

    def decode_pcm_device(self, d_pcm_ptr: int, fmt: str, n_channels: int, channel: int, track_stride_bytes: int, n_samples: int,
                          n_tracks: int, d_audio_ptr: int, audio_stride: int, stream: int | None = None):
        self._check(self.lib.fx_decode_pcm_device(self._h, d_pcm_ptr, PCM_FORMATS[fmt], n_channels, channel, track_stride_bytes,
                                                  n_samples, n_tracks, d_audio_ptr, audio_stride, stream), "fx_decode_pcm_device")

    # -- batch analysis, device buffers (raw pointers; torch is only used by callers for allocation) ----------
    def analyse_device(self, d_audio_ptr: int, track_stride: int, n_samples: int, d_raw_ptr=None, d_smooth_ptr=None,
                       d_diag_ptr=None, stream: int | None = None, d_spec_ptr=None) -> int:
        """d_spec_ptr: device buffer of [n_tracks][frames][window // 2] fp32 (16-byte aligned) that receives the spectrum the
        spectral features read (fx_analyse_device_spectrum); None: no spectrum."""
        nf = c_long(0)
        if d_spec_ptr is None:
            st = self.lib.fx_analyse_device(self._h, d_audio_ptr, track_stride, n_samples, d_raw_ptr, d_smooth_ptr,
                                            d_diag_ptr, stream, ctypes.byref(nf))
            self._check(st, "fx_analyse_device")
        else:
            st = self.lib.fx_analyse_device_spectrum(self._h, d_audio_ptr, track_stride, n_samples, d_raw_ptr, d_smooth_ptr,
                                                     d_diag_ptr, d_spec_ptr, stream, ctypes.byref(nf))
            self._check(st, "fx_analyse_device_spectrum")
        return nf.value

    def synth_device(self, d_audio_ptr: int, track_stride: int, n_samples: int, first_track: int = 0, seed: int = 0x5EED,
                     stream: int | None = None, first_sample: int = 0):
        """Synthetic workload (SURVEY.md 8d): samples [first_sample, first_sample + n_samples) of tracks first_track ..."""
        self._check(self.lib.fx_synth_device_at(self._h, d_audio_ptr, track_stride, n_samples, first_track, first_sample, seed, stream),
                    "fx_synth_device_at")

    # -- real-time path ----------------------------------------------------------------------------------------
    def push_block(self, block: np.ndarray, first_track: int = 0):
        """block: float32 [n_tracks_in_block, n_samples]; row i feeds track first_track + i."""
        b = np.ascontiguousarray(block, dtype=np.float32)
        n, s = b.shape
        ptrs = (c_void_p * n)(*[b.ctypes.data + i * s * 4 for i in range(n)])
        self._check(self.lib.fx_push_block(self._h, first_track, n, ptrs, s), "fx_push_block")

    def process(self) -> int:
        nf = c_long(0)
        self._check(self.lib.fx_process(self._h, ctypes.byref(nf)), "fx_process")
        return nf.value

    def poll(self, track: int):
        out = (c_float * NUM_FEATURES)()
        idx = c_uint64(0)
        self._check(self.lib.fx_poll_features(self._h, track, out, ctypes.byref(idx)), "fx_poll_features")
        return np.frombuffer(out, dtype=np.float32).copy(), idx.value

    def poll_block(self, first_track: int = 0, n_tracks: int | None = None):
        n = self.cfg.n_tracks - first_track if n_tracks is None else n_tracks
        out = np.empty((n, NUM_FEATURES), np.float32)
        idx = np.zeros(n, np.uint64)
        self._check(self.lib.fx_poll_block(self._h, first_track, n, out.ctypes.data, idx.ctypes.data), "fx_poll_block")
        return out, idx

    def rt_start(self, callback=None):
        """Start the group workers.  callback(first_track, n_tracks, frame_index, n_new) runs on a worker thread."""
        if callback is not None:
            self._cb = FEATURES_CALLBACK(lambda user, t0, n, idx, new: callback(t0, n, idx, new))
            self._check(self.lib.fx_set_features_callback(self._h, self._cb, None), "fx_set_features_callback")
        self._check(self.lib.fx_rt_start(self._h), "fx_rt_start")

    def rt_stop(self):
        self._check(self.lib.fx_rt_stop(self._h), "fx_rt_stop")

    def rt_stats(self, reset: bool = False) -> dict:
        s = RtStats()
        self._check(self.lib.fx_rt_get_stats(self._h, ctypes.byref(s), 1 if reset else 0), "fx_rt_get_stats")
        return {k: getattr(s, k) for k, _ in RtStats._fields_}

    def osc_encode(self, tracks, addresses, n_floats: int = 12, stride: int = 128):
        """One OSC 1.0 datagram per listed track from the latest published vectors: list of bytes."""
        n = len(tracks)
        tr = (c_int * n)(*tracks)
        ad = (c_char_p * n)(*[a.encode() for a in addresses])
        out = np.zeros((n, stride), np.uint8)
        sizes = (c_int * n)()
        self._check(self.lib.fx_osc_encode_tracks(self._h, tr, n, ad, n_floats, out.ctypes.data, stride, sizes), "fx_osc_encode_tracks")
        return [out[i, : sizes[i]].tobytes() for i in range(n)]

    def flush(self):
        self._check(self.lib.fx_flush(self._h), "fx_flush")

    def profile_enable(self, on: bool = True):
        self._check(self.lib.fx_profile_enable(self._h, 1 if on else 0), "fx_profile_enable")

    def profile_read(self):
        """(ms in k_analyse, ms in the post kernels, bracketed calls) since the last read"""
        a, b, n = c_double(0), c_double(0), c_long(0)
        self._check(self.lib.fx_profile_read(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(n)), "fx_profile_read")
        return a.value, b.value, n.value

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.fx_kernel_launches(self._h))


def shard_tracks(n_tracks: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous track range [first, first + count) of `rank` when n_tracks are sharded over world_size GPUs.
    Tracks are independent (AnalyserTrackController owns all per-track state, AnalyserTrackController.h:199-210),
    so the multi-GPU path is a partition with no exchange step."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("bad world_size / rank")
    base, extra = divmod(n_tracks, world_size)
    first = rank * base + min(rank, extra)
    return first, base + (1 if rank < extra else 0)


def measure_fp32_peak(device: int = 0) -> float:
    lib = load_library()
    tf = c_double(0)
    st = lib.fx_measure_fp32_peak(device, ctypes.byref(tf))
    if st != 0:
        raise FxError(f"fx_measure_fp32_peak failed ({st})")
    return tf.value


def legacy_analyse(audio: np.ndarray, n_frames: int, window: int = 2048, sample_rate: float = 48000.0, device: int = 0):
    """The legacy offline analyser (AudioAnalysis.h AudioAnalyser) on the GPU: audio float32 [n_tracks, n_samples] ->
    (features [n_tracks, n_frames, 12] in LEGACY order, log attack time [n_tracks])."""
    lib = load_library()
    a = np.ascontiguousarray(np.atleast_2d(audio), dtype=np.float32)
    T, S = a.shape
    out = np.zeros((T, n_frames, len(LEGACY)), np.float32)
    la = np.zeros(T, np.float32)
    st = lib.fx_legacy_analyse_host(device, window, sample_rate, a.ctypes.data, S, S, T, n_frames, out.ctypes.data, la.ctypes.data)
    if st != 0:
        raise FxError(f"fx_legacy_analyse_host failed ({st})")
    return out, la


def h2d_probe(device: int = 0, nbytes: int = 1 << 30, reps: int = 4, write_combined: bool = False) -> float:
    """GB/s of plain pinned -> device cudaMemcpyAsync on `device` (fx_h2d_probe)."""
    lib = load_library()
    g = c_double(0)
    st = lib.fx_h2d_probe(device, nbytes, reps, 1 if write_combined else 0, ctypes.byref(g))
    if st != 0:
        raise FxError(f"fx_h2d_probe failed ({st})")
    return g.value


def osc_order(vec12: np.ndarray, n_out: int = 12) -> np.ndarray:
    lib = load_library()
    v = np.ascontiguousarray(vec12, dtype=np.float32)
    out = np.empty(n_out, np.float32)
    st = lib.fx_osc_order(v.ctypes.data_as(POINTER(c_float)), out.ctypes.data_as(POINTER(c_float)), n_out)
    if st != 0:
        raise FxError(f"fx_osc_order failed ({st})")
    return out

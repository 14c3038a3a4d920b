/*
 * fx_engine.h -- C ABI of the B200-native per-frame analysis engine (libfxb200.so).
 *
 * This is the drop-in boundary for the reference's hot path L1a..L2 (SURVEY.md section 8b):
 * everything between AudioDataCollector::audioDeviceIOCallback (Source/AudioDataCollector.h:36)
 * and AudioFeatures::getValue (Source/RealTimeAnalyser.h:84).  The reference has no FFI of its own --
 * its boundary is the C++ surface of those classes -- so each entry point below cites the reference
 * interface it replaces; feature-extractor_b200/host/ rebuilds that C++ surface (same class names and
 * method signatures) on top of these calls, and INTEGRATION.md shows the binding a maintainer adds.
 *
 * Plain pointers and sizes only; no exceptions cross this boundary; every call returns fx_status
 * (0 = OK, negative = error) and fx_last_error() gives the text.  There is NO CPU fallback: if the
 * CUDA device or kernels are unavailable, fx_engine_create fails.
 *
 * All file:line citations are relative to /root/reference/Source/.
 */
#ifndef FX_ENGINE_H
#define FX_ENGINE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fx_engine fx_engine;
typedef int fx_status;

enum {
    FX_OK                =  0,
    FX_ERR_INVALID_ARG   = -1,
    FX_ERR_CUDA          = -2,
    FX_ERR_UNSUPPORTED   = -3,   /* window not in {1024, 2048, 4096}, hop not a multiple of 16 dividing the window, ... */
    FX_ERR_OVERRUN       = -4,   /* fx_push_block would overwrite samples that were not analysed yet */
    FX_ERR_NO_DEVICE     = -5
};

/* Feature slots: AudioFeatures::eAudioFeature (RealTimeAnalyser.h:17-32). */
enum {
    FX_ONSET = 0, FX_RMS, FX_F0, FX_CENTROID, FX_SPREAD, FX_FLATNESS, FX_LER, FX_FLUX,
    FX_SLOPE, FX_HER, FX_OER, FX_INHARM, FX_NUM_FEATURES
};

/* Per-frame diagnostics: integer decisions and the smallest relative margin that decided them
 * (BASELINE.json north_star: "frames whose decision margin falls below that tolerance ... are counted and reported"). */
enum {
    FX_DIAG_TRUE_OER = 0,    /* log-mapped odd/even ratio (HarmonicCharacteristics.h:190-195); the reference stores HER in its slot (RealTimeAnalyser.h:171) */
    FX_DIAG_LAG,             /* integer pitch lag (PitchAnalyser.h:161-190) */
    FX_DIAG_PITCH_MARGIN,
    FX_DIAG_NUM_PEAKS,       /* HarmonicCharacteristics.h:115-145 */
    FX_DIAG_PEAK_MARGIN,
    FX_DIAG_FLAT_COUNT,      /* bins gated into the flatness product (SpectralCharacteristics.h:89-94) */
    FX_DIAG_FLAT_MARGIN,
    FX_DIAG_GATE_MARGIN,     /* silence gates 0.05 / 0.005 / 1e-4 (SpectralCharacteristics.h:121-123,165-167; HarmonicCharacteristics.h:88) */
    FX_DIAG_ONSET_MARGIN,    /* SpectralCharacteristics.h:271-292 */
    FX_DIAG_FLAT_STATE,      /* 0 finite, 1 product underflowed to 0, 2 overflowed to inf, 3 frame gated silent */
    FX_NUM_DIAG
};

/* The order OSCFeatureAnalysisOutput::sendSpectralFeaturesViaOSC puts on the wire (OSCFeatureAnalysisOutput.h:107):
 * onset, rms, f0, centroid, slope, spread, flatness, ler, flux, her, oer, inharm (12 floats);
 * README.md:55-57 documents the same list without ler and oer (10 floats). */
#define FX_OSC_FLOATS_CODE   12
#define FX_OSC_FLOATS_README 10

/* Spectrum mode (fx_config.spectrum).  The reference squares only the REAL part of each FFT bin wherever it reads a spectrum
 * (SpectralCharacteristics.h:68-73, :158-159; HarmonicCharacteristics.h:63-64; PitchAnalyser.h:100-103), so its features
 * depend on the phase at which the hop meets the signal: a steady tone makes the harmonic energy ratio, inharmonicity,
 * flatness and slope flicker over their whole range.
 *   FX_SPECTRUM_RE_SQUARED  the reference's values (parity mode, the default).
 *   FX_SPECTRUM_POWER       each of the three forward transforms per hop hands its consumers (|X[k]|, 0) in place of
 *                           (Re X[k], Im X[k]), k = 0 .. N-1, |X| = (float) sqrt ((double) Re^2 + (double) Im^2) (the GPU
 *                           forms it in fp32).  Nothing else changes, so the reference's own code defines the result: the
 *                           per-bin value of the spectral features, flux, flatness, slope and harmonic features becomes
 *                           |X|^2; the pitch path's P[k] becomes |C[k]|^2, whose inverse transform is then the true circular
 *                           autocorrelation; the slope's pre-max scans |X[k]| for k < N/4; the previous spectrum holds |X|.
 * The mode applies to every analysis path (fx_analyse_host / _device / _host_pcm and the real-time workers); the legacy
 * analyser is unaffected (it already uses true magnitudes).  fx_engine_create refuses any other value. */
enum { FX_SPECTRUM_RE_SQUARED = 0, FX_SPECTRUM_POWER = 1 };

typedef struct fx_config {
    int    n_tracks;            /* one AnalyserTrackController per track (AnalyserTrackController.h:17) */
    int    window;              /* N: 1024, 2048 (reference: AnalyserTrackController.h:20-21) or 4096 */
    int    hop;                 /* H: reference N/2 (RealTimeAudioAnalysis.h:207); any multiple of 16 dividing N */
    double sample_rate;         /* RealTimeAnalyser.h:100, sampleRateChanged :111-114 */
    int    device;              /* CUDA device ordinal */
    int    rms_pushes_per_frame;/* 2 = both analyser bodies push RMS (RealTimeAnalyser.h:150,209), 1 = spectral only */
    int    onset_type;          /* OnsetDetector::eOnsetDetectionType (SpectralCharacteristics.h:213-219), default 1 = amplitude */
    int    onset_hist;          /* SpectralCharacteristics.h:237-239, default 5, <= 16 */
    float  onset_multiplier;    /* meanThresholdMultiplier, SpectralCharacteristics.h:311, default 1.7 */
    float  gain;                /* AudioDataCollector::setGain (AudioDataCollector.h:124), default 1 */
    long   max_frames_per_call; /* capacity of the engine-owned device result buffers (frames per track per call) */
    int    ring_hops;           /* streaming: device + pinned ring length in hops per track (>= window/hop + 2); 0 = no real-time path */
    int    tracks_per_group;    /* streaming: tracks per CUDA stream / pinned-ring group; 0 = all tracks in one group */
    int    spectrum;            /* FX_SPECTRUM_*: what every spectrum consumer reads per bin; fixed for the engine's life */
} fx_config;
/* NOTE: fx_config grew by the trailing `spectrum` field.  Always fill it with fx_default_config (never a hand-sized
 * copy): a caller compiled against the older, shorter struct has fx_default_config write past its end. */

void        fx_default_config (fx_config* cfg);

/* Replaces constructing AnalyserTrackController x n_tracks (AnalyserTrackController.h:17-45) + prepareToPlay (:175-188). */
fx_status   fx_engine_create  (const fx_config* cfg, fx_engine** out);
fx_status   fx_engine_destroy (fx_engine* e);
const char* fx_last_error     (const fx_engine* e);      /* e may be NULL: last create error */
const char* fx_version        (void);

/* Runtime parameter surface (applies from the next analysed hop; a gain change keeps the older part of the overlapped
 * window at the gain it was collected with, as AudioDataCollector::getAnalysisBuffer applies it on the way out of the
 * ring, AudioDataCollector.h:88).
 * AudioDataCollector::setGain (AudioDataCollector.h:124);
 * RealTimeSpectralAnalyser::setOnsetDetectionType / setOnsetWindowLength / setOnsetDetectionSensitivity
 * (RealTimeAnalyser.h:244-258; multiplier = 1 + sensitivity).  track = -1 applies to every track.
 * As in the reference, changing the window length clears the onset histories. */
fx_status   fx_set_gain  (fx_engine* e, int track, float gain);
fx_status   fx_set_onset (fx_engine* e, int track, int type, int hist_len, float multiplier);

/* Forget all per-track state (overlap buffer, previous spectrum, feature and onset histories): a fresh
 * RealTimeAudioDataOverlapper (RealTimeAudioAnalysis.h:197-203), SpectralCharacteristicsAnalyser
 * (SpectralCharacteristics.h:34-38) and AudioFeatures (RealTimeAnalyser.h:70-74). */
fx_status   fx_reset (fx_engine* e);

/* ---- offline / batch analysis: tracks x frames in one call ---------------------------------------
 * Analyses the NEXT n_samples of every track (state carries over from earlier calls; call fx_reset
 * for a fresh stream).  audio is [n_tracks][track_stride] fp32; frames = n_samples / hop per track.
 * Outputs are [n_tracks][frames][12] raw (values as pushed into AudioFeatures::updateFeature,
 * RealTimeAnalyser.h:76), [n_tracks][frames][12] smoothed (AudioFeatures::getValue, :84-88, after both
 * analyser bodies of the hop) and [n_tracks][frames][FX_NUM_DIAG]; any may be NULL.
 *
 * Only complete hops are analysed: n_samples % hop trailing samples are not carried over (pass them again at the head of
 * the next call).  The offline calls are refused while the real-time workers run, and need the track groups in step
 * (they are unless the real-time path advanced them independently; fx_reset brings them back).
 *
 * fx_analyse_host: HOST pointers (pinned or pageable); host<->device copies are inside the call,
 *                  pipelined over track groups; returns when the results are in host memory.
 * fx_analyse_device: DEVICE pointers, asynchronous on `stream` (a cudaStream_t; NULL = the engine's own). */
fx_status   fx_analyse_host   (fx_engine* e, const float* audio, long track_stride, long n_samples,
                               float* raw, float* smooth, float* diag, long* n_frames);
fx_status   fx_analyse_device (fx_engine* e, const float* d_audio, long track_stride, long n_samples,
                               float* d_raw, float* d_smooth, float* d_diag, void* stream, long* n_frames);

/* fx_analyse_device_spectrum: fx_analyse_device that also writes the spectrum the spectral features are computed from.
 * d_spec is DEVICE memory, [n_tracks][frames][window / 2] fp32, contiguous: 2 * window bytes per track and frame (15.7 GB
 * for 4096 tracks x 10 s at 48 kHz, N = 4096, H = 1024).  Row (t, f), bin m = 0 .. window/2 - 1 holds mag[m], the value
 * SpectralCharacteristics.h:68-73 reads for frame f, rounded once to fp32:
 *   FX_SPECTRUM_RE_SQUARED  (Re X[m])^2
 *   FX_SPECTRUM_POWER       |X[m]|^2
 * where X is the transform of the Bartlett-windowed frame with the gain applied (after a gain change the older part of the
 * window keeps its old gain, as for the features).  Every frame is written, the ones the 0.05 magnitude gate silences and
 * the zero-padded start of a stream included.  d_spec must be 16-byte aligned (FX_ERR_INVALID_ARG otherwise, nothing
 * written); d_spec = NULL is fx_analyse_device.  The output is device-only: copying it to the host would take several
 * times as long as the analysis. */
fx_status   fx_analyse_device_spectrum (fx_engine* e, const float* d_audio, long track_stride, long n_samples,
                                        float* d_raw, float* d_smooth, float* d_diag, float* d_spec,
                                        void* stream, long* n_frames);

/* ---- file ingest: PCM in, features out ---------------------------------------------------------------
 * Replaces the file route of the reference: AudioFilePlayer::loadFileIntoTransport (AudioFilePlayer.h:41-60) hands the
 * file to JUCE's format readers, the transport plays it through the device output and AudioDataCollector re-captures one
 * output channel (AudioDataCollector.h:42-43).  Here the bytes of the file's data chunk go to the GPU as they are
 * (interleaved sample frames, WAV little endian / AIFF big endian), kernel k_pcm_decode converts the one channel each
 * track analyses to fp32 exactly as JUCE's readers do ((float) left-justified int32 * (1.0f / 0x7fffffff); 8-bit WAV is
 * offset binary; float data passes through), and the analysis runs on the result.  Integer samples of <= 24 bits
 * convert exactly, so a 16-bit file crosses PCIe at 2 bytes per sample and still yields the fp32 input the
 * float API would have been given. */
enum {
    FX_PCM_U8 = 1, FX_PCM_S8, FX_PCM_S16LE, FX_PCM_S16BE, FX_PCM_S24LE, FX_PCM_S24BE,
    FX_PCM_S32LE, FX_PCM_S32BE, FX_PCM_F32LE, FX_PCM_F32BE
};
int         fx_pcm_bytes_per_sample (int format);        /* 0 for an unknown format */
/* pcm holds n_tracks rows, track_stride_bytes apart; each row is n_samples sample frames of n_channels interleaved
 * samples, of which `channel` is analysed.  channel = -1: track t analyses channel t % n_channels (the reference's
 * tracks each pick one channel of the same device stream); track_stride_bytes = 0: every track reads the same row (one
 * multichannel file feeding all tracks).  Otherwise as fx_analyse_host (HOST pointers, pipelined copies, state carries
 * over).  fx_decode_pcm_device is the conversion alone on DEVICE pointers, asynchronous on `stream`. */
fx_status   fx_analyse_host_pcm  (fx_engine* e, const void* pcm, int format, int n_channels, int channel,
                                  long track_stride_bytes, long n_samples,
                                  float* raw, float* smooth, float* diag, long* n_frames);
fx_status   fx_decode_pcm_device (fx_engine* e, const void* d_pcm, int format, int n_channels, int channel,
                                  long track_stride_bytes, long n_samples, long n_tracks,
                                  float* d_audio, long audio_stride, void* stream);

/* ---- real-time path --------------------------------------------------------------------------------
 * Threading contract (SURVEY.md section 8b; the reference: AudioDataCollector.h:36-70 only copies and notifies, the
 * analysis runs on two juce::Threads per track, RealTimeAnalyser.h:97-127, AnalyserTrackController.h:184-185):
 *
 *   audio thread      fx_push_block ONLY.  Wait-free: bounds check, memcpy into the pinned ring, one atomic publish per
 *                     track and -- when a hop became complete and the group's worker is asleep -- one futex wake.  No lock,
 *                     no allocation, no CUDA call.  One producer thread per track at a time.
 *   worker threads    one per track group, inside the engine (fx_rt_start / fx_rt_stop): sleeps until a hop is complete on
 *                     every ACTIVE track of its group, streams the new samples to the device (cudaMemcpyAsync on the
 *                     group's stream), analyses them, brings the smoothed vectors back and publishes them under a
 *                     seqlock; then calls the features callback.  Groups advance independently of each other.
 *   any other thread  fx_poll_features / fx_poll_block / fx_osc_encode_tracks (lock-free snapshots, never torn);
 *                     the parameter calls fx_set_gain / fx_set_onset / fx_set_sample_rate / fx_set_track_active /
 *                     fx_clear_buffer / fx_reset (they take the affected groups' batch mutex, i.e. they are applied
 *                     between two batches = at a hop boundary; the audio thread never touches that mutex).
 *
 * Every device and host buffer of this path is sized at fx_engine_create for ring_hops hops: the steady state performs no
 * allocation and no device-wide synchronisation.  ring_hops = 0 creates the engine without the real-time path.
 *
 * fx_push_block replaces AudioDataCollector::audioDeviceIOCallback (AudioDataCollector.h:36-70) for a range of tracks;
 * channels[i] is track first_track + i.  FX_ERR_OVERRUN: a block did not fit (the analysis fell behind by a whole ring);
 * NOTHING of the call was copied, the overrun is counted (fx_rt_stats) and the tracks stay in step.  Blocks for inactive
 * tracks are dropped.
 * fx_process is the synchronous form of one worker pass over every group, on the calling thread -- a test hook and the
 * way to drive the engine without worker threads; it must not be called while the workers run (FX_ERR_INVALID_ARG).
 * fx_poll_features replaces AudioFeatures::getValue x 12 as read by the OSC / GUI timers (OSCFeatureAnalysisOutput.h:91-104). */
fx_status   fx_push_block    (fx_engine* e, int first_track, int n_tracks, const float* const* channels, int n_samples);
fx_status   fx_process       (fx_engine* e, long* n_new_frames);
fx_status   fx_poll_features (fx_engine* e, int track, float out12[FX_NUM_FEATURES], uint64_t* frame_index);
/* the same for a range of tracks in one call: out [n_tracks][12], frame_index [n_tracks] (may be NULL) */
fx_status   fx_poll_block    (fx_engine* e, int first_track, int n_tracks, float* out, uint64_t* frame_index);
fx_status   fx_flush         (fx_engine* e);             /* synchronise every group stream */

/* juce::Thread::startThread / stopThread of the analysers (AnalyserTrackController.h:184-185,190-194) for the whole engine:
 * start the group workers / stop and join them (idempotent). */
fx_status   fx_rt_start      (fx_engine* e);
fx_status   fx_rt_stop       (fx_engine* e);
/* Called on a worker thread after the features of `n_new` hops of tracks [first_track, first_track + n_tracks) were
 * published (frame_index = hops analysed so far in that group) -- where RealTimeSpectralAnalyser::run fires its
 * onsetDetectedCallback (RealTimeAnalyser.h:228-229).  Set it before fx_rt_start. */
/* The callback may read (fx_poll_*, fx_osc_encode_tracks, fx_rt_get_stats); it must not call the parameter, start / stop or
 * analysis entry points (they wait for the workers). */
typedef void (*fx_features_callback) (void* user, int first_track, int n_tracks, uint64_t frame_index, int n_new);
fx_status   fx_set_features_callback (fx_engine* e, fx_features_callback cb, void* user);
/* A track is what one AnalyserTrackController owns (AnalyserTrackController.h:17-45).  Only active tracks gate their
 * group's progress; an inactive track is fed silence.  Activating with reset_state != 0 gives the track the state of a
 * freshly constructed controller (zero overlap buffer, zero previous spectrum, empty feature / onset histories) starting at
 * the group's current hop.  All tracks are active after fx_engine_create.  track = -1: every track. */
fx_status   fx_set_track_active (fx_engine* e, int track, int active, int reset_state);
/* AudioDataCollector::clearBuffer (AudioDataCollector.h:122, fired by play / pause / stop / file drop,
 * AnalyserTrackController.h:131-133,167-171, and by toggleCollectInput :119): the samples pushed but not analysed yet
 * (and the rest of the ring) become zeros; positions do not move. */
fx_status   fx_clear_buffer  (fx_engine* e, int track);
/* RealTimeAnalyser::sampleRateChanged -> FFTAnalyser::setNyquistValue (RealTimeAnalyser.h:111-114, called for both
 * analysers on every prepareToPlay, AnalyserTrackController.h:178-179): every frequency-dependent quantity (bin
 * frequencies, f0 = 2 nyquist / lag, the harmonic bin tables) follows from the next analysed hop on. */
fx_status   fx_set_sample_rate (fx_engine* e, double sample_rate);

typedef struct fx_rt_stats {
    uint64_t batches;            /* worker passes that analysed at least one hop (all groups) */
    uint64_t hops;               /* hops analysed (summed over groups) */
    uint64_t overruns;           /* fx_push_block calls refused */
    double   batch_ms_mean;      /* wake-up -> features published, per batch */
    double   batch_ms_max;
} fx_rt_stats;
fx_status   fx_rt_get_stats  (fx_engine* e, fx_rt_stats* out, int reset);

/* ---- OSC wire output (OSCFeatureAnalysisOutput.h:89-113) -----------------------------------------------
 * Batch encoder: for each listed track one complete OSC 1.0 message -- address pattern addresses[i] (the reference's
 * bundleAddress, "/Audio/A<n>", MainComponent.cpp:170), type tags ",f" x n_floats, n_floats big-endian floats of the latest
 * published vector in the order of :107 (n_floats = 12) or README.md:55-57 (10) -- written at out + i * datagram_stride;
 * sizes[i] receives its length (0 when it would not fit the stride).  One pass over the published block; the caller sends
 * the datagrams (the facade: one sendmmsg per 60 Hz tick). */
fx_status   fx_osc_encode_tracks (fx_engine* e, const int* tracks, int n_tracks, const char* const* addresses, int n_floats,
                                  unsigned char* out, int datagram_stride, int* sizes);

/* OSC argument order (OSCFeatureAnalysisOutput.h:107): reorder one 12-slot feature vector.
 * n_out = 12 (as the code sends) or 10 (as README.md:55-57 documents). */
fx_status   fx_osc_order (const float in12[FX_NUM_FEATURES], float* out, int n_out);

/* ---- legacy offline analyser (SURVEY.md section 8 row f4) ----------------------------------------------------
 * struct AudioAnalyser of AudioAnalysis.h: the per-frame pipeline of performSpectralAnalysis (:121-251) with the feature
 * block that the reference has commented out at its own call site (:219-247) reinstated -- frame i centred on sample
 * i * stepSize (stepSize = n_samples / n_frames, :130), zero padded, symmetric Bartlett ramps (:663-672), TRUE magnitudes
 * of bins 0 .. N/2 (performFrequencyOnlyForwardTransform :208, :226-227), then calculateSpectralCharacteristics (:463-515),
 * calculateNormalisedSpectralSlope (:566-609), calculateHarmonicCharacteristics (:253-306: histogram of peak intervals,
 * previousF0 hysteresis :279-298, inharmonicity :308-338), the energy envelope (:249), analyseNormalisedZeroCrosses (:517-541)
 * and setLogAttackTime (:611-622).  The application never instantiates AudioAnalyser; this entry point exists for callers
 * of that class.  audio is [n_tracks][track_stride] fp32 HOST memory (one channel per track); out is
 * [n_tracks][n_frames][FX_LEGACY_NUM]; log_attack [n_tracks] (may be NULL).  Self-contained: needs no fx_engine. */
enum {
    FX_LEGACY_CENTROID = 0,   /* centroid / nyquist (:514) */
    FX_LEGACY_SPREAD, FX_LEGACY_FLATNESS, FX_LEGACY_FLUX, FX_LEGACY_SLOPE,
    FX_LEGACY_F0,             /* Hz, after the previousF0 rule */
    FX_LEGACY_HER, FX_LEGACY_INHARM,
    FX_LEGACY_ZCR,            /* zero crossings * 2 / stepSize (:538) */
    FX_LEGACY_ENERGY,         /* energy envelope (:249) */
    FX_LEGACY_NUM_PEAKS,      /* diagnostic: peak bins of the frame (:366-387) */
    FX_LEGACY_PRODUCT_STATE,  /* diagnostic: the ungated fp64 product (:491): 0 finite, 1 reached 0, 2 reached inf, 3 ended denormal, 4 frame silent */
    FX_LEGACY_NUM
};
fx_status   fx_legacy_analyse_host (int device, int window, double sample_rate, const float* audio, long track_stride,
                                    long n_samples, int n_tracks, int n_frames, float* out, float* log_attack);

/* ---- measurement support (bench.py; not part of the reference surface) -------------------------------
 * Fill d_audio [n_tracks][track_stride] with the synthetic workload of SURVEY.md section 8d:
 * A sin(2 pi f_t n / sr + phi_t) + sigma_t u_t[n], Philox-4x32-10 keyed by (seed, track), with the
 * silence / burst insertions.  first_track offsets the track index (multi-GPU sharding by track range). */
fx_status   fx_synth_device (fx_engine* e, float* d_audio, long track_stride, long n_samples,
                             long first_track, uint64_t seed, void* stream);
/* the same for samples [first_sample, first_sample + n_samples) of every track: the generator is a pure function of
 * (seed, track, sample index), so a long stream can be produced slab by slab without a seam */
fx_status   fx_synth_device_at (fx_engine* e, float* d_audio, long track_stride, long n_samples,
                                long first_track, long first_sample, uint64_t seed, void* stream);
/* number of kernels this engine has launched since creation */
uint64_t    fx_kernel_launches (const fx_engine* e);
/* Per-kernel device timing: when enabled, every call brackets the analysis kernel (k_analyse) and the small
 * post kernels with CUDA events on the stream they are launched on.  fx_profile_read synchronises those events
 * and returns the accumulated milliseconds and the number of bracketed calls since the last read. */
fx_status   fx_profile_enable (fx_engine* e, int on);
fx_status   fx_profile_read   (fx_engine* e, double* ms_analyse, double* ms_post, long* n_calls);
/* FP32 FMA microbenchmark (registers only) for the compute roofline denominator: achieved TFLOP/s on `device`. */
fx_status   fx_measure_fp32_peak (int device, double* tflops);
/* Host -> device link probe: `reps` cudaMemcpyAsync of `bytes` from a pinned (optionally write-combined) host buffer,
 * GB/s by CUDA events.  Run on every rank at once it measures the box's concurrent upload ceiling. */
fx_status   fx_h2d_probe (int device, long bytes, int reps, int write_combined, double* gbs);

#ifdef __cplusplus
}
#endif
#endif

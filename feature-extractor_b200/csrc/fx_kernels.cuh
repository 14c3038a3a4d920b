// fx_kernels.cuh -- kernel parameter blocks and launch entry points shared by fx_analyse.cu,
// fx_post.cu and fx_engine.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/fx_engine.h"

namespace fx {

constexpr int kHistRows   = 32;   // raw feature rows carried between calls (10-tap smoothing + <=16-deep onset window + 5)
constexpr int kMaxOnsetHist = 16;
#define FX_HER_TAB_STRIDE 20       // shorts per lag in AnalyseParams::her_tab

// What K1 leaves for K1b (k_finalize) per frame: a FrameHead followed by one WarpPart per warp of the K1 CTA (window / 512 of
// them), frame_rec_bytes (window) per frame.  fp64 wherever the reference accumulates in double.
// The sums that only K1b looks at leave K1 as PER-WARP partials, stored by each warp where it forms them (one 80-byte run per
// warp): K1 reduces across warps only what its own threads need (magnitude sum, maxima, the lag search), and no warp collects
// the others' partials on its way into the next frame's first barrier (-2.4 % kernel time at N = 2048 / 1024, where the five
// parts of the old record stage shared four / two warps).  K1b adds them in the order of the butterfly K1 used to run
// (pairwise tree over the warps), so the features are the same bits.  The raw moments of pass 1 cross the lanes of their warp
// in fp64, because K1b's spread is a cancelling difference of them (fx_analyse.cu); the other partials (flux, low-energy and
// gated sums, the inharmonicity sum, the mantissa of the flatness product's scan) are reduced in fp32 and stored as such: an
// 80-byte WarpPart, and a frame record of 304 / 464 / 784 bytes at N = 1024 / 2048 / 4096.
struct alignas (16) WarpPart
{
    double p1d[4];      // pass 1, fp64 slots: S0 = sum mag, W1 = sum x mag, S2 = sum x^2 mag, S4 = sum mag^2     (x = (bin + 1/2) / M)
    float  p1f[3];      // pass 1, fp32 slots: flux, low-energy sum, gated sum
    float  inharm;      // sum of f0Proportion * binMagnitude over the warp's peaks
    float  scan_m;      // extended-range product of the warp's gated magnitudes: mantissa in [0.5, 1] ...
    int    scan_e;      // ... and exponent
    int    count;       // gated bins
    int    npeaks;
    float  rawmax;      // max |Re|, |Im| of the lower bins (slope quirk)
};
struct alignas (16) FrameHead
{
    double rms_sum, mag_sum, maxmag, product, hsum, hmax;
    float  flat_state;             // 3: silent frame, 0 / 1 / 2: product finite / 0 / inf after a range event (K1 replayed it), -1: no event, K1b multiplies the warp products
    float  have_prev, lag, pitch_margin, peak_margin, flat_margin;
    float  her_mx[18];             // largest |Re A| around the 15 sub-octave and 3 harmonic bins of f0 (HarmonicCharacteristics.h:147-210), < 0: not used
};
static_assert (sizeof (WarpPart) == 80 && sizeof (FrameHead) == 144, "the records are runs of 16-byte multiples (bulk copies in K1b)");
__host__ __device__ constexpr size_t frame_rec_bytes (int window) { return sizeof (FrameHead) + (size_t) (window / 512) * sizeof (WarpPart); }

// ---- K1: per-(track, chunk) frame walker ------------------------------------------------------------
struct AnalyseParams
{
    // source: this call's samples, [n_tracks][track_stride]; hop block b (0-based in this call) at b * hop
    const float* audio;
    long         track_stride;
    // carry-in / carry-out overlap tail, [n_tracks][window - hop] (the last window/hop - 1 hop blocks of the stream)
    const float* tail_in;
    float*       tail_out;
    long         first_hop;        // absolute hop index (since stream start) of this call's hop block 0
    int          n_frames;         // frames (= hop blocks) per track in this call
    int          frames_per_chunk;
    int          n_chunks;
    int          hop;
    int          log2_hop;
    int          use_bulk;         // 1: cp.async.bulk (16-byte aligned source), 0: plain loads
    int          want_margins;     // 1: the decision margins (diagnostics) are computed as well; 0: the instantiation without them
    const float* gain;             // [n_tracks]
    double       sample_rate;
    double       bin_var;          // slope: sum ((i/M - 0.5)^2) / M evaluated on the host in the reference's order
    float        iir_c1, iir_c2;   // pi/2 and exp (-pi/2) in fp32 (RealTimeAudioAnalysis.h:122)
    const float2* tw2;             // stage-2 twiddles, the full table (fx_fft.cuh layout): K1 copies the rows k2 = 1, 2, 4, 8
    const float2* tw1f;            // stage-1 twiddles in full, [(k1 - 1) * 256 + m] = W_N^(m k1) (the two-factor product, rounded as the kernel used to), read through L1
    // per-lag tables, slot lag = 1 .. window, slot 0 = "no lag found" (lag -1), evaluated on the host in the reference's own
    // double arithmetic from f0 = (nyquist * 2) / lag (PitchAnalyser.h:57):
    // her_tab[lag][0..14] = bin of the sub-octave f0 / 2^(l+1), [15..17] = bin of the harmonic h f0, h = 1..3, or -1 when the
    // reference does not use it (HarmonicCharacteristics.h:158-185); [18] = bin of f0 itself (:246-249), clamped to a short
    const short*  her_tab;
    const double* ex_tab;          // inharmonicity fractions of the (lag, bin) pairs with exact-integer edge ratios (fx_engine.cu: build_exact_ratio_table)
    const int*    ex_off;          // [window + 1] offset of a lag's entries in ex_tab
    short        f0bin_pow2[16];   // her_tab[lag][18] for lag = 2^k (the lags whose f0 bin the kernel does not derive by integer division)
    // outputs
    unsigned char* rec;            // [n_tracks][n_frames] records of frame_rec_bytes (window) each
    float*       first_spec;       // [n_tracks][n_chunks][M]  Re (power mode: |X|) spectrum (windowed path) of the chunk's first non-silent frame
    float*       last_spec;        // [n_tracks][n_chunks][M]  ... of its last non-silent frame
    int*         first_idx;        // [n_tracks][n_chunks]     frame index of the first non-silent frame, -1 if none
    int          spectrum;         // fx_config::spectrum: FX_SPECTRUM_RE_SQUARED or FX_SPECTRUM_POWER (selects the instantiation)
    // (last, so that the offsets of the fields above -- and the instructions of the kernels without it -- stay as they were)
    float*       spec;             // [n_tracks][n_frames][M] mag[m] of every frame, 16-byte aligned, 64-bit row index; null: not exported (selects the instantiation)
};

int         analyse_ctas_per_sm (int window);      // resident CTAs per SM k_analyse is compiled for (chunk heuristic)
cudaError_t launch_analyse (int window, long n_tracks, const AnalyseParams& p, cudaStream_t stream);
cudaError_t configure_analyse (int window);             // opt in to the dynamic shared memory the kernel needs
size_t      analyse_smem_bytes (int window);

// ---- K1b: scalar tail (pow / log10 / sqrt, gates, clamps), one thread per frame --------------------
struct FinalizeParams
{
    const unsigned char* rec;      // [n_rows] records of frame_rec_bytes (window)
    long         n_rows;           // n_tracks * n_frames
    int          window;
    double       sample_rate;
    double       bin_var;
    float*       raw;              // [n_rows][12]
    float*       diag;             // [n_rows][FX_NUM_DIAG] (may be null)
};
cudaError_t launch_finalize (const FinalizeParams& p, cudaStream_t stream);

// ---- K2: flux of each chunk's first non-silent frame against the carried previous spectrum ----------
struct FluxFixParams
{
    int          n_frames, n_chunks, m;   // m = window / 2
    const float* first_spec;
    const float* last_spec;
    const int*   first_idx;
    const float* prev_in;          // [n_tracks][M] carried "previousBinMagnitudes" as Re values, |X| in power mode (zeros after reset)
    float*       prev_out;
    float*       raw;
};
cudaError_t launch_flux_fix (long n_tracks, const FluxFixParams& p, cudaStream_t stream);

// ---- K3: AudioFeatures smoothing + OnsetDetector, a FIR along frames --------------------------------
struct SmoothParams
{
    int          n_frames;
    long         frames_before;    // frames analysed since stream start before this call
    int          rms_pushes;
    float*       raw;              // onset slot is written here
    float*       smooth;           // [n_tracks][n_frames][12] (may be null)
    float*       diag;             // onset margin written here (may be null)
    const float* hist_in;          // [n_tracks][kHistRows][12], newest row last
    float*       hist_out;
    const int*   onset_type;       // [n_tracks]
    const int*   onset_hist;
    const float* onset_mult;
    const long*  onset_reset;      // [n_tracks] absolute frame index at which the onset histories were last cleared
    const long*  track_start;      // [n_tracks] absolute frame index at which the track's own stream started (may be null: 0)
    float*       latest;           // [n_tracks][12 + 2] smoothed vector of the newest frame + 64-bit frame count as two words (may be null)
};
cudaError_t launch_smooth (long n_tracks, const SmoothParams& p, cudaStream_t stream);

// ---- K0: file ingest, interleaved PCM -> track-major fp32 (fx_pcm.cu) ----------------------------------
struct PcmParams
{
    const unsigned char* pcm;      // [n_tracks] rows of interleaved sample frames, track_stride_bytes apart
    long         track_stride_bytes;
    int          format;           // FX_PCM_*
    int          n_channels;       // samples per frame in the source
    int          channel;          // the one channel each track analyses (AudioDataCollector.h:42-43); -1: track t takes channel (first_track + t) % n_channels
    long         first_track;      // engine index of row 0 (only used by channel == -1)
    long         n_samples;        // frames to decode per track
    long         n_tracks;
    float*       audio;            // [n_tracks][audio_stride]
    long         audio_stride;
};
cudaError_t launch_pcm_decode (const PcmParams& p, cudaStream_t stream);
int         pcm_launch_count (const PcmParams& p);
__host__ __device__ inline int pcm_bytes_per_sample (int format)
{
    switch (format)
    {
        case FX_PCM_U8: case FX_PCM_S8:                                               return 1;
        case FX_PCM_S16LE: case FX_PCM_S16BE:                                         return 2;
        case FX_PCM_S24LE: case FX_PCM_S24BE:                                         return 3;
        case FX_PCM_S32LE: case FX_PCM_S32BE: case FX_PCM_F32LE: case FX_PCM_F32BE:   return 4;
        default:                                                                      return 0;
    }
}

// ---- synthetic workload ------------------------------------------------------------------------------
cudaError_t launch_synth (float* d_audio, long track_stride, long n_samples, long n_tracks, long first_track, long first_sample,
                          double sample_rate, uint64_t seed, cudaStream_t stream);

// ---- gain change between calls: rescale the carried overlap of the tracks whose ratio is not 1 ----------
cudaError_t launch_tail_scale (float* tail, long tail_len, const float* ratio, long n_tracks, cudaStream_t stream);

// ---- FP32 FMA microbenchmark ---------------------------------------------------------------------------
cudaError_t measure_fp32_peak (double* tflops);

} // namespace fx

// fx_post.cu -- the small kernels around K1 (sm_100a):
//   K2  k_flux_fix   flux of each chunk's first non-silent frame against the carried previous spectrum, and the
//                    carry-out of "previousBinMagnitudes" (SpectralCharacteristics.h:75-79, :121-123, :138)
//   K3  k_smooth     AudioFeatures / ValueHistory moving averages (RealTimeAnalyser.h:70-88,
//                    RealTimeAudioAnalysis.h:40-96) and OnsetDetector (SpectralCharacteristics.h:243-306)
//       k_hist       carry the last raw rows to the next call
//       k_tail_scale a gain change between calls: carried overlap rescaled to the gain it was collected at
//       k_synth      synthetic workload generator (SURVEY.md section 8d) -- measurement support only
// All citations relative to /root/reference/Source/.
#include "fx_kernels.cuh"
#include <math.h>

namespace fx {

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__ (256) k_flux_fix (const FluxFixParams p)
{
    const long cta = blockIdx.x;
    const int chunk = (int) (cta % p.n_chunks);
    const long track = cta / p.n_chunks;
    const int t = threadIdx.x;
    const int M = p.m;
    const int* fidx = p.first_idx + track * p.n_chunks;

    __shared__ double wsum[8];

    int last_chunk = -1;                       // last chunk of this call holding a non-silent frame
    for (int c = p.n_chunks - 1; c >= 0; --c) if (fidx[c] >= 0) { last_chunk = c; break; }

    // carry-out: the newest non-silent spectrum of the track
    if (chunk == (last_chunk >= 0 ? last_chunk : 0))
    {
        const float* from = last_chunk >= 0 ? p.last_spec + (track * p.n_chunks + last_chunk) * (long) M
                                            : p.prev_in + track * (long) M;
        float* to = p.prev_out + track * (long) M;
        for (int i = t; i < M; i += blockDim.x) to[i] = from[i];
    }

    const int fi = fidx[chunk];
    if (fi < 0) return;

    const float* prev = p.prev_in + track * (long) M;
    for (int c = chunk - 1; c >= 0; --c)
        if (fidx[c] >= 0) { prev = p.last_spec + (track * p.n_chunks + c) * (long) M; break; }
    const float* cur = p.first_spec + (track * p.n_chunks + chunk) * (long) M;

    // The sum runs in K1's own order and precision, so that a frame's flux does not depend on where the chunk boundaries fall
    // (tests: chunked, streamed and split calls are bit-identical): thread t takes bins 8 t .. 8 t + 7 in sequence (fp64), the
    // lanes of a warp are added as K1's butterfly does (distances 1, 2, 4, 8, 16; in fp32 like K1's) and
    // the warps as K1b's pairwise tree.  blockDim.x = M / 8 = the thread count of K1.
    double flux = 0.0;
    {
        const float4 c0 = *reinterpret_cast<const float4*> (cur + 8 * t), c1 = *reinterpret_cast<const float4*> (cur + 8 * t + 4);
        const float4 q0 = *reinterpret_cast<const float4*> (prev + 8 * t), q1 = *reinterpret_cast<const float4*> (prev + 8 * t + 4);
        const float cv[8] = { c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w }, qv[8] = { q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w };
        #pragma unroll
        for (int j = 0; j < 8; ++j)
        {
            const double c = (double) cv[j], q = (double) qv[j];
            const double diff = c * c - q * q;                        // SpectralCharacteristics.h:76 (both products are exact)
            if (diff > 0.0) flux += diff;                             // :77-79
        }
    }
    float fl = (float) flux;
    #pragma unroll
    for (int off = 1; off < 32; off <<= 1) fl += __shfl_xor_sync (0xffffffffu, fl, off);
    flux = (double) fl;
    if ((t & 31) == 0) wsum[t >> 5] = flux;
    __syncthreads();
    if (t == 0)
    {
        const int nw = (int) (blockDim.x >> 5);
        for (int half = 1; half < nw; half <<= 1)
            for (int w = 0; w < nw; w += 2 * half) wsum[w] += wsum[w + half];
        const float max_flux = (float) (M * (M + 1)) / 2.0f;          // :111
        p.raw[(track * p.n_frames + fi) * FX_NUM_FEATURES + FX_FLUX] = (float) (wsum[0] / (double) max_flux);
    }
}

cudaError_t launch_flux_fix (long n_tracks, const FluxFixParams& p, cudaStream_t stream)
{
    const long grid = n_tracks * p.n_chunks;
    if (grid <= 0) return cudaSuccess;
    k_flux_fix<<<(unsigned) grid, (unsigned) (p.m / 8), 0, stream>>> (p);     // one thread per 8 bins, like K1
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ const float* raw_row (const SmoothParams& p, long track, long j)
{
    const long rel = j - p.frames_before;
    if (rel >= 0) return p.raw + (track * p.n_frames + rel) * FX_NUM_FEATURES;
    return p.hist_in + (track * kHistRows + (kHistRows + rel)) * FX_NUM_FEATURES;
}

// smoothed RMS as RealTimeSpectralAnalyser::detectOnset reads it (RealTimeAnalyser.h:239): after the spectral
// body's push of frame j, before the harmonic body's
__device__ __forceinline__ float amp_at_spectral_time (const SmoothParams& p, long track, long j, long start)
{
    float total = 0.0f;
    const long jr = j - start;                                  // frames of this track before frame j
    if (p.rms_pushes >= 2)
    {
        if (j - 5 >= start) total += raw_row (p, track, j - 5)[FX_RMS];
        for (long q = j - 4; q < j; ++q)
            if (q >= start) { const float r = raw_row (p, track, q)[FX_RMS]; total += r; total += r; }
        total += raw_row (p, track, j)[FX_RMS];
        const long rec = 2 * jr + 1 < 10 ? 2 * jr + 1 : 10;
        return total / (float) (int) rec;
    }
    for (long q = j - 9; q <= j; ++q)
        if (q >= start) total += raw_row (p, track, q)[FX_RMS];
    const long rec = jr + 1 < 10 ? jr + 1 : 10;
    return total / (float) (int) rec;
}

__device__ __forceinline__ float relmarginf (float a, float b)
{
    const float m = fmaxf (fabsf (a), fabsf (b));
    return (m > 0.0f) ? fabsf (a - b) / m : 0.0f;
}

__global__ void __launch_bounds__ (128) k_smooth (const SmoothParams p, long n_tracks)
{
    const long idx = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_tracks * p.n_frames) return;
    const long track = idx / p.n_frames;
    const int f = (int) (idx % p.n_frames);
    const long g = p.frames_before + f;                       // absolute frame index of the track group's stream
    // hop at which this track's own stream started (a controller created while the engine runs): earlier frames do not
    // exist for it -- fresh ValueHistory objects have recorded nothing (RealTimeAudioAnalysis.h:40-96)
    const long start = p.track_start ? p.track_start[track] : 0;
    float* row = p.raw + (track * p.n_frames + f) * FX_NUM_FEATURES;

    // ---- onset (spectral body, after the flux / RMS pushes of frame g) -----------------------------------
    const int L = p.onset_hist[track];
    const int type = p.onset_type[track];
    const float mult = p.onset_mult[track];
    float onset = 0.0f, om = 1.0f;
    const long onset_from = p.onset_reset[track] > start ? p.onset_reset[track] : start;
    if (g - onset_from + 1 >= L)                              // SpectralCharacteristics.h:253-258: histories full
    {
        float am[kMaxOnsetHist], sf[kMaxOnsetHist];
        float tot_am = 0.0f, tot_sf = 0.0f;
        for (int i = 0; i < L; ++i)
        {
            const long j = g - L + 1 + i;
            am[i] = amp_at_spectral_time (p, track, j, start);
            sf[i] = 0.0f + raw_row (p, track, j)[FX_FLUX];    // depth-1 history: getValue = (0 + v) / 1
            tot_am += am[i];                                  // ValueHistory::getTotal, oldest first
            tot_sf += sf[i];
        }
        const float mean_sf = tot_sf / (float) L, mean_am = tot_am / (float) L;           // :260-261
        int cand = L - 1;                                                                 // :263
        if (type == 0 || type == 2) cand = L / 2;                                         // :265-266
        const float cand_sf = sf[cand], cand_am = am[cand];
        bool ok = true;
        om = fminf (om, relmarginf (cand_am, 0.01f));
        if (cand_am < 0.01f) ok = false;                                                  // :271-274
        for (int i = 0; ok && i < L; ++i)
        {
            if (i == cand) continue;
            if (type == 1 || type == 2) { om = fminf (om, relmarginf (am[i], cand_am)); if (am[i] >= cand_am) ok = false; }    // :283
            if (ok && (type == 0 || type == 2)) { om = fminf (om, relmarginf (sf[i], cand_sf)); if (sf[i] >= cand_sf) ok = false; }   // :286
        }
        if (ok)
        {
            const bool o_sf = cand_sf > mean_sf * mult, o_am = cand_am > mean_am * mult;  // :291-292
            if (type != 0) om = fminf (om, relmarginf (cand_am, mean_am * mult));
            if (type != 1) om = fminf (om, relmarginf (cand_sf, mean_sf * mult));
            const bool on = (type == 1) ? o_am : (type == 0 ? o_sf : (type == 2 ? (o_am && o_sf) : false));
            onset = on ? 1.0f : 0.0f;
        }
    }
    row[FX_ONSET] = onset;
    if (p.diag) p.diag[(track * p.n_frames + f) * FX_NUM_DIAG + FX_DIAG_ONSET_MARGIN] = om;

    // ---- AudioFeatures::getValue for every slot, after both analyser bodies of frame g -------------------
    // Every history is summed oldest value first like ValueHistory::getTotal.  The ten rows of the window are read once, as
    // three 16-byte loads each (a row is 48 bytes), and added to the twelve running totals in that order: 30 loads instead of
    // 120 (the kernel is bound by its load instructions: 0.32 -> 0.1x ms per 1.9e6 rows).
    float sm[FX_NUM_FEATURES];
    const long gr = g - start;                                // frames of this track before this one
    const long rec10 = gr + 1 < 10 ? gr + 1 : 10;
    float tot[FX_NUM_FEATURES];
    #pragma unroll
    for (int k = 0; k < FX_NUM_FEATURES; ++k) tot[k] = 0.0f;
    float rms2 = 0.0f;                                        // RMS with two pushes per frame: the last five frames, twice each
    #pragma unroll 1
    for (long q = g - 9; q <= g; ++q)
    {
        if (q < start) continue;
        const float4* r4 = reinterpret_cast<const float4*> (raw_row (p, track, q));
        const float4 a = r4[0], b = r4[1], c = r4[2];
        const float rv[FX_NUM_FEATURES] = { a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w };
        #pragma unroll
        for (int k = 0; k < FX_NUM_FEATURES; ++k) tot[k] += rv[k];
        if (q >= g - 4) { rms2 += rv[FX_RMS]; rms2 += rv[FX_RMS]; }
    }
    #pragma unroll
    for (int k = 0; k < FX_NUM_FEATURES; ++k)
    {
        if (k == FX_ONSET)      sm[k] = (0.0f + onset) / 1.0f;
        else if (k == FX_FLUX)  sm[k] = (0.0f + row[FX_FLUX]) / 1.0f;                     // depth 1 (RealTimeAnalyser.h:73)
        else if (k == FX_RMS && p.rms_pushes >= 2)
        {
            const long rec = 2 * (gr + 1) < 10 ? 2 * (gr + 1) : 10;
            sm[k] = rms2 / (float) (int) rec;
        }
        else sm[k] = tot[k] / (float) (int) rec10;                                        // :84-88
    }
    if (p.smooth)
    {
        float* so = p.smooth + (track * p.n_frames + f) * FX_NUM_FEATURES;
        for (int k = 0; k < FX_NUM_FEATURES; ++k) so[k] = sm[k];
    }
    if (p.latest && f == p.n_frames - 1)
    {
        float* lo = p.latest + track * (FX_NUM_FEATURES + 2);
        for (int k = 0; k < FX_NUM_FEATURES; ++k) lo[k] = sm[k];
        const unsigned long long cnt = (unsigned long long) (gr + 1);      // hops of this track analysed so far
        lo[FX_NUM_FEATURES]     = __uint_as_float ((unsigned) (cnt & 0xffffffffull));
        lo[FX_NUM_FEATURES + 1] = __uint_as_float ((unsigned) (cnt >> 32));
    }
}

__global__ void __launch_bounds__ (128) k_hist (const SmoothParams p, long n_tracks)
{
    const long idx = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_tracks * kHistRows * FX_NUM_FEATURES) return;
    const int k = (int) (idx % FX_NUM_FEATURES);
    const int i = (int) ((idx / FX_NUM_FEATURES) % kHistRows);
    const long track = idx / (FX_NUM_FEATURES * kHistRows);
    const long j = p.frames_before + p.n_frames - kHistRows + i;
    float v = 0.0f;
    const long start = p.track_start ? p.track_start[track] : 0;
    if (j >= start && j >= p.frames_before - kHistRows) v = raw_row (p, track, j)[k];
    p.hist_out[(track * kHistRows + i) * FX_NUM_FEATURES + k] = v;
}

cudaError_t launch_smooth (long n_tracks, const SmoothParams& p, cudaStream_t stream)
{
    const long total = n_tracks * p.n_frames;
    if (total > 0)
    {
        k_smooth<<<(unsigned) ((total + 127) / 128), 128, 0, stream>>> (p, n_tracks);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    const long ht = n_tracks * kHistRows * FX_NUM_FEATURES;
    k_hist<<<(unsigned) ((ht + 127) / 128), 128, 0, stream>>> (p, n_tracks);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// A gain change between two calls: the overlap carried in `tail` was collected at the old gain (AudioDataCollector.h:88
// multiplies on the way out of the ring, so the older part of the next windows keeps it) while K1 applies the track's
// current gain to the whole window.  Scaling the carried samples by old / new once restores the reference's mixed-gain
// windows up to two fp32 roundings per sample.
__global__ void __launch_bounds__ (256) k_tail_scale (float* tail, long tail_len, const float* __restrict__ ratio)
{
    const float r = ratio[blockIdx.x];
    if (r == 1.0f) return;
    float* row = tail + (long) blockIdx.x * tail_len;
    for (long i = threadIdx.x; i < tail_len; i += blockDim.x) row[i] *= r;
}

cudaError_t launch_tail_scale (float* tail, long tail_len, const float* ratio, long n_tracks, cudaStream_t stream)
{
    if (n_tracks <= 0 || tail_len <= 0) return cudaSuccess;
    k_tail_scale<<<(unsigned) n_tracks, 256, 0, stream>>> (tail, tail_len, ratio);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// Philox-4x32-10 (Salmon et al. 2011), counter = sample index / 4, key = seed ^ track
__device__ __forceinline__ void philox4x32_10 (uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out)
{
    #pragma unroll
    for (int r = 0; r < 10; ++r)
    {
        const uint32_t hi0 = __umulhi (0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi (0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// sin (2 pi r) for r in [0, 1) from IEEE double add / multiply only (explicit _rn intrinsics: no FMA contraction), so that
// the test suite reproduces every sample bit for bit with numpy (tests: synth_tracks): quadrant q = floor (4 r + 1/2),
// z = r - q / 4 in [-1/8, 1/8], Taylor polynomials of sin / cos in a = 2 pi z (|a| <= pi / 4: truncation < 1e-11).
__device__ __forceinline__ double synth_sin_turns (double r)
{
    const double q = floor (__dadd_rn (__dmul_rn (4.0, r), 0.5));
    const double z = __dadd_rn (r, -__dmul_rn (0.25, q));
    const double a = __dmul_rn (z, 6.283185307179586);
    const double a2 = __dmul_rn (a, a);
    double ps = -2.505210838544172e-08;                                                   // -1/11!
    ps = __dadd_rn (__dmul_rn (ps, a2),  2.755731922398589e-06);                          //  1/9!
    ps = __dadd_rn (__dmul_rn (ps, a2), -1.984126984126984e-04);                          // -1/7!
    ps = __dadd_rn (__dmul_rn (ps, a2),  8.333333333333333e-03);                          //  1/5!
    ps = __dadd_rn (__dmul_rn (ps, a2), -1.666666666666667e-01);                          // -1/3!
    ps = __dadd_rn (__dmul_rn (ps, a2),  1.0);
    const double sn = __dmul_rn (a, ps);
    double pc = -2.755731922398589e-07;                                                   // -1/10!
    pc = __dadd_rn (__dmul_rn (pc, a2),  2.480158730158730e-05);                          //  1/8!
    pc = __dadd_rn (__dmul_rn (pc, a2), -1.388888888888889e-03);                          // -1/6!
    pc = __dadd_rn (__dmul_rn (pc, a2),  4.166666666666666e-02);                          //  1/4!
    pc = __dadd_rn (__dmul_rn (pc, a2), -0.5);
    pc = __dadd_rn (__dmul_rn (pc, a2),  1.0);
    const int qi = ((int) q) & 3;
    return qi == 0 ? sn : (qi == 1 ? pc : (qi == 2 ? -sn : -pc));
}

struct SynthFreqs { double f[48]; };     // 110 * 2^(k / 12), evaluated on the host (exp2 is not correctly rounded everywhere)

__global__ void __launch_bounds__ (256) k_synth (float* audio, long track_stride, long n_samples, long n_tracks,
                                                 long first_track, long first_sample, double sample_rate, uint64_t seed, const SynthFreqs fr)
{
    // first_sample is a multiple of 4: one Philox block yields the four samples 4 c .. 4 c + 3 of the stream
    const long quads = (n_samples + 3) / 4;
    const long idx = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_tracks * quads) return;
    const long tl = idx / quads;
    const long i0 = (idx % quads) * 4;                                                    // index inside this call's buffer
    const long n0 = first_sample + i0;                                                    // index inside the stream
    const long track = first_track + tl;
    const uint64_t key = seed ^ (uint64_t) track;
    uint32_t r[4];
    philox4x32_10 ((uint32_t) (n0 >> 2), (uint32_t) ((uint64_t) (n0 >> 2) >> 32), 0u, 0u, (uint32_t) key, (uint32_t) (key >> 32), r);

    const int reg = (int) (track & 7);
    const double sigma = reg == 6 ? 0.5 : (reg == 7 ? 0.001 : 0.05);                      // the three flatness regimes (SURVEY Q7)
    const double freq = fr.f[track % 48];
    double ph = __dmul_rn ((double) track, 0.61803398874989484820);
    ph = __dadd_rn (ph, -floor (ph));                                                     // phi_t / (2 pi)
    const long sr = (long) sample_rate;
    float* dst = audio + tl * track_stride;
    #pragma unroll
    for (int i = 0; i < 4; ++i)
    {
        const long n = n0 + i;
        if (i0 + i >= n_samples) break;
        const double u = __dadd_rn (__dmul_rn ((double) (r[i] >> 8), 1.0 / 8388608.0), -1.0);   // uniform [-1, 1), exact
        double turns = __dadd_rn (__ddiv_rn (__dmul_rn (freq, (double) n), sample_rate), ph);
        turns = __dadd_rn (turns, -floor (turns));
        double x = __dadd_rn (__dmul_rn (0.5, synth_sin_turns (turns)), __dmul_rn (sigma, u));
        if ((n % sr) < sr / 20) x = __dmul_rn (x, 4.0);                                   // burst at the top of every second (onsets)
        if ((track & 1) && (n % (2 * sr)) >= sr && (n % (2 * sr)) < sr + sr / 4) x = 0.0; // 0.25 s of silence every 2 s on odd tracks
        dst[i0 + i] = (float) x;
    }
}

cudaError_t launch_synth (float* d_audio, long track_stride, long n_samples, long n_tracks, long first_track, long first_sample,
                          double sample_rate, uint64_t seed, cudaStream_t stream)
{
    const long total = n_tracks * ((n_samples + 3) / 4);
    if (total <= 0) return cudaSuccess;
    if (first_sample & 3) return cudaErrorInvalidValue;
    SynthFreqs fr;
    for (int k = 0; k < 48; ++k) fr.f[k] = 110.0 * pow (2.0, (double) k / 12.0);
    k_synth<<<(unsigned) ((total + 255) / 256), 256, 0, stream>>> (d_audio, track_stride, n_samples, n_tracks, first_track, first_sample, sample_rate, seed, fr);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// 8 independent FMA chains per thread, 2 flops per FMA; enough CTAs to fill every SM several times over
__global__ void __launch_bounds__ (256) k_fma_peak (float* sink, int iters, float a, float b)
{
    float r0 = threadIdx.x * 1e-3f, r1 = r0 + 1.0f, r2 = r0 + 2.0f, r3 = r0 + 3.0f, r4 = r0 + 4.0f, r5 = r0 + 5.0f, r6 = r0 + 6.0f, r7 = r0 + 7.0f;
    for (int i = 0; i < iters; ++i)
    {
        #pragma unroll
        for (int u = 0; u < 16; ++u)
        {
            r0 = fmaf (r0, a, b); r1 = fmaf (r1, a, b); r2 = fmaf (r2, a, b); r3 = fmaf (r3, a, b);
            r4 = fmaf (r4, a, b); r5 = fmaf (r5, a, b); r6 = fmaf (r6, a, b); r7 = fmaf (r7, a, b);
        }
    }
    const float s = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    if (s == 123.456f) sink[0] = s;
}

cudaError_t measure_fp32_peak (double* tflops)
{
    cudaDeviceProp prop{};
    int dev = 0;
    cudaError_t e = cudaGetDevice (&dev);
    if (e != cudaSuccess) return e;
    e = cudaGetDeviceProperties (&prop, dev);
    if (e != cudaSuccess) return e;
    float* sink = nullptr;
    e = cudaMalloc (&sink, 64);
    if (e != cudaSuccess) return e;
    cudaEvent_t a, b;
    cudaEventCreate (&a); cudaEventCreate (&b);
    const int blocks = prop.multiProcessorCount * 16, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep)
    {
        cudaEventRecord (a);
        k_fma_peak<<<blocks, 256>>> (sink, iters, 0.999f, 1e-4f);
        cudaEventRecord (b);
        e = cudaEventSynchronize (b);
        if (e != cudaSuccess) break;
        float ms = 0.0f;
        cudaEventElapsedTime (&ms, a, b);
        const double flops = (double) blocks * 256.0 * (double) iters * 16.0 * 8.0 * 2.0;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy (a); cudaEventDestroy (b);
    cudaFree (sink);
    *tflops = best;
    return e;
}

} // namespace fx

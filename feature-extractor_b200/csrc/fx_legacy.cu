// fx_legacy.cu -- the legacy offline analyser (SURVEY.md section 8 row f4) on the GPU, sm_100a.
//
// Replaces struct AudioAnalyser of /root/reference/Source/AudioAnalysis.h: the per-frame pipeline of performSpectralAnalysis
// (:121-251) with the feature block that the reference has commented out at its own call site (:219-247) reinstated, i.e.
// calculateSpectralCharacteristics (:463-515, TRUE magnitudes, ungated fp64 product), calculateNormalisedSpectralSlope
// (:566-609), calculateHarmonicCharacteristics (:253-306: histogram of peak intervals, previousF0 hysteresis, inharmonicity),
// the energy envelope (:249), analyseNormalisedZeroCrosses (:517-541) and setLogAttackTime (:611-622).
// The application never instantiates AudioAnalyser; parity is checked against those member functions driven headless
// (oracle/ref_driver.cpp: fxo_legacy_analyse).  All citations below are AudioAnalysis.h lines.
//
// Kernels (grid = tracks x frames unless noted):
//   L1 k_legacy_spectrum   frame centred on sample i * stepSize, zero padded, symmetric Bartlett ramps (:145-181), the shared-
//                          memory FFT of fx_fft.cuh, magnitudes (float) sqrt (re^2 + im^2) of bins 0 .. N/2 (:208, :226-227)
//   L2 k_legacy_prev       (one thread per track) index of the last non-silent frame before each frame: previousBinMagnitudes
//                          is only overwritten when magnitudeSum > 0.001 (:497-498 returns before :508)
//   L3 k_legacy_features   spectral characteristics, slope, energy, peak bins, interval histogram, best candidate
//   L4 k_legacy_hysteresis (one thread per track) the previousF0 rule (:279-298) along the frames, log attack time
//   L5 k_legacy_inharm     inharmonicity of the frame's peaks against the final f0 (:308-338)
//   L6 k_legacy_zcr        zero crossings of the frame's step (:517-541)
#include "fx_fft.cuh"
#include "fx_kernels.cuh"
#include "fx_tables.h"
#include <math.h>
#include <vector>

namespace fx {

namespace {

struct LegacyRec            // per frame, L3 -> L4 / L5
{
    double sum;             // magnitudeSum (:262-266)
    double f0, her;         // best histogram candidate (:415-436), then the final values after L4
    float  energy;          // :249
    int    n_peaks;
};

struct LegacyParams
{
    const float* audio; long track_stride, n_samples;
    int n_frames, step, nb, nbp;          // nb = N / 2 + 1 bins, nbp = padded row length of `mags`
    double sample_rate, bin_var;
    float* mags;                          // [tracks][frames][nbp]
    double* fsum;                         // [tracks][frames]
    int* prev_idx;                        // [tracks][frames]
    LegacyRec* rec;                       // [tracks][frames]
    float* out;                           // [tracks][frames][FX_LEGACY_NUM]
    float* log_attack;                    // [tracks]
    const float2* tw1f; const float2* tw2;
};

__device__ __forceinline__ double block_sum (double v, double* sh)
{
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync (0xffffffffu, v, off);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += sh[w];
    return t;
}
__device__ __forceinline__ float block_maxf (float v, double* sh)
{
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = fmaxf (v, __shfl_xor_sync (0xffffffffu, v, off));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = (double) v;
    __syncthreads();
    float t = 0.0f;
    for (int w = 0; w < nw; ++w) t = fmaxf (t, (float) sh[w]);
    return t;
}

// ---- L1 ---------------------------------------------------------------------------------------------------------
template <int R1>
__global__ void __launch_bounds__ (16 * R1) k_legacy_spectrum (const LegacyParams p)
{
    using D = FftDims<R1>;
    constexpr int N = D::N, T = D::T, Q1 = D::Q1;
    __shared__ float2 ex[D::EX_LEN];
    __shared__ float2 tw2[D::TW2_FULL];
    __shared__ double red[8];
    const int t = threadIdx.x;
    const long row = blockIdx.x;
    const long track = row / p.n_frames;
    const int frame = (int) (row % p.n_frames);
    for (int i = t; i < D::TW2_FULL; i += T) tw2[i] = p.tw2[i];
    const float* src = p.audio + track * p.track_stride;
    // :150-161: the window is centred on sample frame * stepSize unless the whole signal is one frame
    const long origin = p.n_frames == 1 ? 0 : (long) frame * p.step - N / 2;
    float2 v[16];
    #pragma unroll
    for (int q = 0; q < Q1; ++q)
        #pragma unroll
        for (int n1 = 0; n1 < R1; ++n1)
        {
            const int n = n1 * 256 + t + T * q;
            const long k = origin + n;
            float x = (k >= 0 && k < p.n_samples) ? src[k] : 0.0f;                         // :169-177 zero padding
            // scaleBufferWithBartlettWindowing (:663-672): applyGainRamp 0 -> 1 over the first half, 1 -> 0 over the second;
            // the gain is accumulated additively in fp32, which is exact for these power-of-two steps
            const float g = n < N / 2 ? (float) n * (2.0f / N) : 1.0f - (float) (n - N / 2) * (2.0f / N);
            v[q * R1 + n1] = make_float2 (__fmul_rn (x, g), 0.0f);
        }
    __syncthreads();
    fft_stage1_store<R1, false> (v, t, ex, p.tw1f);
    __syncthreads();
    fft_stage2<R1, false, false> (t, ex, tw2);
    __syncwarp();
    fft_stage3<R1, false> (t, ex);
    __syncthreads();
    // :208 performFrequencyOnlyForwardTransform: juce_hypot per bin; :226-227 the first N / 2 + 1 of them
    float* mg = p.mags + row * p.nbp;
    double sum = 0.0;
    for (int k = t; k < p.nb; k += T)
    {
        const float2 z = ex[zpos<R1> (k)];
        const float m = (float) sqrt ((double) z.x * (double) z.x + (double) z.y * (double) z.y);
        mg[k] = m;
        sum += (double) m;
    }
    sum = block_sum (sum, red);
    if (t == 0) p.fsum[row] = sum;
}

// ---- L2 ---------------------------------------------------------------------------------------------------------
__global__ void k_legacy_prev (const LegacyParams p, long n_tracks)
{
    const long track = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (track >= n_tracks) return;
    int last = -1;
    for (int f = 0; f < p.n_frames; ++f)
    {
        p.prev_idx[track * p.n_frames + f] = last;
        if (p.fsum[track * p.n_frames + f] > 0.001) last = f;                              // :497-498 / :508
    }
}

// extended-range product of non-negative doubles: value = m * 2^e, m in [0.5, 1)
struct LME { double m; int e; };
__device__ __forceinline__ LME lme_from (double x)
{
    LME r;
    int e;
    r.m = frexp (x, &e);
    r.e = e;
    return r;
}
__device__ __forceinline__ LME lme_mul (LME a, LME b)
{
    LME r;
    r.m = a.m * b.m; r.e = a.e + b.e;
    if (r.m < 0.5) { r.m *= 2.0; r.e -= 1; }
    return r;
}

__device__ __forceinline__ bool legacy_is_peak (const float* mg, int nb, int bin, double mean)          // binIsPeak :366-387
{
    const double m = (double) mg[bin];
    if (m <= mean) return false;
    const int left = bin < 2 ? 2 - bin : 0;
    const int right = bin >= nb - 2 ? 2 - ((nb - 1) - bin) : 0;
    for (int n = bin - (2 - left); n < bin + (2 - right); n++)
        if (n != bin && (double) mg[n] > m) return false;
    return true;
}

// F0Candidate::updateHarmonicEnergyRatio :79-98 (explicit _rn operations: no contraction, as the host compiler's)
__device__ __forceinline__ double legacy_her (const float* mg, int nb, double frequency, double frpb, double total)
{
    double score = 0.0;
    for (int h = 1; h < 16; ++h)
    {
        const double hf = __dmul_rn (frequency, (double) h);
        const int bin = (int) ceil (__ddiv_rn (hf, frpb));
        if (bin >= nb) break;
        score += (double) mg[bin];
    }
    return __ddiv_rn (score, total);
}

// ---- L3 ---------------------------------------------------------------------------------------------------------
constexpr int kLegacyThreads = 256;
constexpr int kLegacyMaxBins = 2049;

__global__ void __launch_bounds__ (kLegacyThreads) k_legacy_features (const LegacyParams p)
{
    __shared__ float mg[kLegacyMaxBins + 3];
    __shared__ int   cnt[kLegacyMaxBins + 3];
    __shared__ int   first[kLegacyMaxBins + 3];
    __shared__ int   peaks[kLegacyMaxBins / 2 + 2];
    __shared__ double red[8];
    __shared__ double scan_m[8];
    __shared__ int scan_e[8], ev_over[8], ev_under[8], ev_zero[8], warp_peaks[8];
    __shared__ double best_w[8]; __shared__ int best_first[8], best_d[8];

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long row = blockIdx.x;
    const long track = row / p.n_frames;
    const int nb = p.nb;
    const double nyquist = p.sample_rate / 2.0;
    const double frpb = nyquist / (double) nb;
    const float* src = p.mags + row * p.nbp;
    const int pi = p.prev_idx[row];
    const float* prev = pi >= 0 ? p.mags + (track * p.n_frames + pi) * p.nbp : nullptr;
    float* o = p.out + row * FX_LEGACY_NUM;

    for (int k = t; k < nb; k += kLegacyThreads) { mg[k] = src[k]; cnt[k] = 0; first[k] = 0x7fffffff; }
    __syncthreads();

    // ---- calculateSpectralCharacteristics :463-515: contiguous bins per thread (the product is order dependent) -------------
    const int per = (nb + kLegacyThreads - 1) / kLegacyThreads;
    const int k0 = t * per, k1 = min (nb, k0 + per);
    double s_sum = 0.0, s_w = 0.0, s_flux = 0.0, s_energy = 0.0;
    float s_max = 0.0f;
    LME prod; prod.m = 0.5; prod.e = 1;
    int zero_at = 0x7fffffff;
    for (int k = k0; k < k1; ++k)
    {
        const double m = (double) mg[k];
        const double fc = (double) k * frpb + (frpb / 2.0);                                // :477
        const double pm = prev ? (double) prev[k] : 0.0;
        const double diff = fabs (m) - fabs (pm);                                          // :482-485
        if (diff > 0.0) s_flux += diff;
        s_sum += m;
        s_w += fc * m;
        s_energy += m;
        s_max = fmaxf (s_max, fabsf (mg[k]));
        if (m == 0.0) zero_at = min (zero_at, k);
        else prod = lme_mul (prod, lme_from (m));
    }
    const double sum = block_sum (s_sum, red);
    const double weighted = block_sum (s_w, red);
    const double flux = block_sum (s_flux, red);
    const float fmx = block_maxf (s_max, red);
    // running product (:491) in bin order: inclusive scan of the per-thread extended-range products; the first prefix that
    // leaves the fp64 range decides what the reference's plain double holds from there on (inf / 0 are sticky)
    LME inc = prod;
    #pragma unroll
    for (int off = 1; off < 32; off <<= 1)
    {
        LME ot; ot.m = __shfl_up_sync (0xffffffffu, inc.m, off); ot.e = __shfl_up_sync (0xffffffffu, inc.e, off);
        if (lane >= off) inc = lme_mul (ot, inc);
    }
    if (lane == 31) { scan_m[warp] = inc.m; scan_e[warp] = inc.e; }
    __syncthreads();
    LME pre; pre.m = 0.5; pre.e = 1;
    for (int w = 0; w < warp; ++w) { LME wt; wt.m = scan_m[w]; wt.e = scan_e[w]; pre = lme_mul (pre, wt); }
    LME excl; excl.m = __shfl_up_sync (0xffffffffu, inc.m, 1); excl.e = __shfl_up_sync (0xffffffffu, inc.e, 1);
    if (lane == 0) { excl.m = 0.5; excl.e = 1; }
    LME run = lme_mul (pre, excl);
    int over_at = 0x7fffffff, under_at = 0x7fffffff;
    for (int k = k0; k < k1; ++k)
    {
        const double m = (double) mg[k];
        if (m == 0.0) continue;
        run = lme_mul (run, lme_from (m));
        if (run.e > 1024) over_at = min (over_at, k);                                      // > DBL_MAX
        if (run.e < -1074) under_at = min (under_at, k);                                   // below half the smallest denormal
    }
    over_at = __reduce_min_sync (0xffffffffu, over_at); under_at = __reduce_min_sync (0xffffffffu, under_at);
    zero_at = __reduce_min_sync (0xffffffffu, zero_at);
    if (lane == 0) { ev_over[warp] = over_at; ev_under[warp] = under_at; ev_zero[warp] = zero_at; }
    __syncthreads();
    LME total; total.m = 0.5; total.e = 1;
    for (int w = 0; w < kLegacyThreads / 32; ++w)
    {
        LME wt; wt.m = scan_m[w]; wt.e = scan_e[w]; total = lme_mul (total, wt);
        over_at = min (over_at, ev_over[w]); under_at = min (under_at, ev_under[w]); zero_at = min (zero_at, ev_zero[w]);
    }
    const double energy = block_sum (s_energy, red);

    float centroid = 0.0f;
    const bool silent = ! (sum > 0.001);                                                   // :496-498
    if (silent) { if (t == 0) { o[FX_LEGACY_CENTROID] = o[FX_LEGACY_SPREAD] = o[FX_LEGACY_FLATNESS] = o[FX_LEGACY_FLUX] = 0.0f; } }
    else centroid = (float) (weighted / sum);                                              // :499
    double s_var = 0.0;
    if (! silent)
        for (int k = k0; k < k1; ++k)
        {
            const double fc = (double) k * frpb + (frpb / 2.0);
            const double dv = (fc / nyquist) - ((double) centroid / nyquist);             // :506 (centroid / nyquist: float / double)
            s_var += (dv * dv) * (double) mg[k];
        }
    const double var = block_sum (s_var, red);
    if (! silent && t == 0)
    {
        // what the reference's double holds after the loop: the first event is sticky; inf * 0 (a zero bin after an overflow) is NaN
        double product; float state = 0.0f;
        const int first_ev = min (over_at, min (under_at, zero_at));
        if (first_ev == 0x7fffffff) product = ldexp (total.m, total.e);
        else if (first_ev == over_at) { product = (zero_at != 0x7fffffff && zero_at > over_at) ? nan ("") : (double) INFINITY; state = 2.0f; }
        else { product = 0.0; state = 1.0f; }
        if (first_ev == 0x7fffffff && total.e < -1021) state = 3.0f;                      // ended in the denormal band: low bits lost in the reference
        const double inv = 1.0 / (double) nb;
        const float flatness = (float) (pow (product, inv) / (inv * sum));                 // :503
        const float max_spread = (float) (((double) centroid / nyquist) * (1.0 - ((double) centroid / nyquist)));      // :510
        o[FX_LEGACY_CENTROID] = centroid / (float) nyquist;                               // :514
        o[FX_LEGACY_SPREAD] = (float) ((var / sum) / (double) max_spread);
        o[FX_LEGACY_FLATNESS] = flatness;
        o[FX_LEGACY_FLUX] = (float) flux;
        o[FX_LEGACY_PRODUCT_STATE] = state;
    }
    if (silent && t == 0) o[FX_LEGACY_PRODUCT_STATE] = 4.0f;

    // ---- calculateNormalisedSpectralSlope :566-609 ------------------------------------------------------------------
    {
        const double fm = (double) fmx;                                                    // getMagnitude :572
        double s_me = 0.0, s_ps = 0.0;
        const bool flat0 = ! (fm > 0.0001);                                                // :574-576
        if (! flat0)
            for (int k = k0; k < k1; ++k) { const double e = (double) mg[k] / fm; s_me += e; s_ps += (double) k * e; }
        double mean_e = block_sum (s_me, red);
        const double prod_sum = block_sum (s_ps, red);
        mean_e /= (double) nb;
        double s_ev = 0.0;
        if (! flat0)
            for (int k = k0; k < k1; ++k) { const double e = (double) mg[k] / fm; s_ev += (e - mean_e) * (e - mean_e); }
        const double ev = block_sum (s_ev, red);
        if (t == 0)
        {
            float slope = 0.0f;
            if (! flat0)
            {
                const double num_bins = (double) nb;
                const double bin_std = sqrt (p.bin_var), energy_std = sqrt (ev / num_bins);
                const double r = (prod_sum - (num_bins * mean_e * 0.5)) / (num_bins - 1.0f) * energy_std * bin_std;   // :603
                slope = (float) (r * (bin_std / energy_std));                              // :606
            }
            o[FX_LEGACY_SLOPE] = slope;
            o[FX_LEGACY_ENERGY] = (float) energy;                                          // :249 (the reference sums in fp32, bin order)
        }
    }

    // ---- calculateHarmonicCharacteristics :253-306, up to the best candidate of the histogram --------------------------
    LegacyRec rec; rec.sum = sum; rec.f0 = 0.0; rec.her = 0.0; rec.energy = (float) energy; rec.n_peaks = 0;
    if (! (sum < 0.001))                                                                   // :270-271
    {
        const double mean = sum / (double) nb;
        // peak bins in bin order (:350-363): flags -> ranks by a block-wide count
        int mine = 0; unsigned flags = 0u;
        for (int k = k0; k < k1; ++k) if (legacy_is_peak (mg, nb, k, mean)) { flags |= 1u << (k - k0); ++mine; }
        int incl = mine;
        #pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const int ov = __shfl_up_sync (0xffffffffu, incl, off); if (lane >= off) incl += ov; }
        if (lane == 31) warp_peaks[warp] = incl;
        __syncthreads();
        int base = incl - mine, n_peaks = 0;
        for (int w = 0; w < kLegacyThreads / 32; ++w) { if (w < warp) base += warp_peaks[w]; n_peaks += warp_peaks[w]; }
        for (int k = k0; k < k1; ++k) if (flags & (1u << (k - k0))) peaks[base++] = k;
        __syncthreads();
        rec.n_peaks = n_peaks;
        // addNewPeakBinAndUpdateHistogram :389-403: every pair (new peak a, earlier peak b) adds one count to interval
        // peaks[a] - peaks[b]; the histogram vector's order is the order of first appearance = the smallest (a, b)
        const long pairs = (long) n_peaks * (n_peaks - 1) / 2;
        for (long q = t; q < pairs; q += kLegacyThreads)
        {
            // q -> (a, b), a > b, enumerated a-major
            int a = (int) ((1.0 + sqrt (1.0 + 8.0 * (double) q)) * 0.5);
            while ((long) a * (a - 1) / 2 > q) --a;
            while ((long) (a + 1) * a / 2 <= q) ++a;
            const int b = (int) (q - (long) a * (a - 1) / 2);
            const int d = peaks[a] - peaks[b];
            atomicAdd (&cnt[d], 1);
            atomicMin (&first[d], a * 4096 + b);
        }
        __syncthreads();
        // estimateF0AndHERFromFrequencyHistogram :415-436: the largest count * harmonicEnergyRatio, the earliest on ties; it
        // must exceed 0
        double bw = 0.0; int bf = 0x7fffffff, bd = 0;
        for (int d = 1 + t; d < nb; d += kLegacyThreads)
        {
            if (cnt[d] == 0) continue;
            const double freq = __dmul_rn ((double) d, frpb);                              // updateFrequency :62-65
            const double w = __dmul_rn ((double) cnt[d], legacy_her (mg, nb, freq, frpb, sum));
            if (w > bw || (w == bw && w > 0.0 && first[d] < bf)) { bw = w; bf = first[d]; bd = d; }
        }
        #pragma unroll
        for (int off = 16; off > 0; off >>= 1)
        {
            const double ow = __shfl_xor_sync (0xffffffffu, bw, off);
            const int of = __shfl_xor_sync (0xffffffffu, bf, off), od = __shfl_xor_sync (0xffffffffu, bd, off);
            if (ow > bw || (ow == bw && ow > 0.0 && of < bf)) { bw = ow; bf = of; bd = od; }
        }
        if (lane == 0) { best_w[warp] = bw; best_first[warp] = bf; best_d[warp] = bd; }
        __syncthreads();
        if (t == 0)
        {
            for (int w = 1; w < kLegacyThreads / 32; ++w)
                if (best_w[w] > bw || (best_w[w] == bw && bw > 0.0 && best_first[w] < bf)) { bw = best_w[w]; bf = best_first[w]; bd = best_d[w]; }
            if (bw > 0.0)
            {
                rec.f0 = __dmul_rn ((double) bd, frpb);
                rec.her = legacy_her (mg, nb, rec.f0, frpb, sum);
            }
        }
    }
    if (t == 0) { p.rec[row] = rec; o[FX_LEGACY_NUM_PEAKS] = (float) rec.n_peaks; }
}

// ---- L4 ---------------------------------------------------------------------------------------------------------
__global__ void k_legacy_hysteresis (const LegacyParams p, long n_tracks)
{
    const long track = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (track >= n_tracks) return;
    const int nb = p.nb;
    const double frpb = (p.sample_rate / 2.0) / (double) nb;
    double previous_f0 = 0.0;                                                              // :107
    float best_e = 0.0f; int best_i = 0;
    for (int f = 0; f < p.n_frames; ++f)
    {
        const long row = track * p.n_frames + f;
        LegacyRec r = p.rec[row];
        float* o = p.out + row * FX_LEGACY_NUM;
        if (f == 0 || r.energy > best_e) { best_e = r.energy; best_i = f; }              // findMinMax + first index equal to the maximum (:615-619)
        if (r.sum < 0.001) { o[FX_LEGACY_F0] = o[FX_LEGACY_HER] = 0.0f; r.f0 = 0.0; p.rec[row] = r; continue; }      // :270-271 (previousF0 untouched)
        double f0 = r.f0, her = r.her;
        if (previous_f0 != f0 && previous_f0 > 10.0)                                       // :279-298
        {
            const double top = previous_f0 > f0 ? previous_f0 : f0;
            const double bottom = top == previous_f0 ? f0 : previous_f0;
            const double ratio = __ddiv_rn (top, bottom);
            if (ratio > 2.0 && ratio - floor (ratio) < 0.1)
            {
                f0 = previous_f0;
                her = legacy_her (p.mags + row * p.nbp, nb, f0, frpb, r.sum);
            }
        }
        previous_f0 = f0;
        r.f0 = f0; r.her = her;
        p.rec[row] = r;
        o[FX_LEGACY_F0] = (float) f0; o[FX_LEGACY_HER] = (float) her;
    }
    // setLogAttackTime :611-622
    const double ms_per_sample = 1.0 / (double) ((int) p.sample_rate / 1000);
    p.log_attack[track] = (float) log10 ((double) (float) (best_i * p.step) * (float) ms_per_sample);
}

// ---- L5 ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double legacy_ratio (double f1, double f2)                      // getFrequencyRatio :340-348
{
    if (f1 == f2) return 1.0;
    const double higher = f1 > f2 ? f1 : f2;
    const double lower = higher == f1 ? f2 : f1;
    return __ddiv_rn (higher, lower);
}

__global__ void __launch_bounds__ (kLegacyThreads) k_legacy_inharm (const LegacyParams p)
{
    __shared__ float mg[kLegacyMaxBins + 3];
    __shared__ double red[8];
    const int t = threadIdx.x;
    const long row = blockIdx.x;
    const LegacyRec r = p.rec[row];
    float* o = p.out + row * FX_LEGACY_NUM;
    if (! (r.f0 > 0.0) || r.sum < 0.001) { if (t == 0) o[FX_LEGACY_INHARM] = 0.0f; return; }      // :302-303
    const int nb = p.nb;
    const double frpb = (p.sample_rate / 2.0) / (double) nb;
    const float* src = p.mags + row * p.nbp;
    for (int k = t; k < nb; k += kLegacyThreads) mg[k] = src[k];
    __syncthreads();
    const double mean = r.sum / (double) nb;
    const int f0_bin = (int) ceil (__ddiv_rn (r.f0, frpb));                                // getBinForFrequency :438-443
    double acc = 0.0;
    for (int bin = t; bin < nb; bin += kLegacyThreads)
    {
        if (! legacy_is_peak (mg, nb, bin, mean) || bin == f0_bin) continue;               // :313-316
        double start = __dmul_rn ((double) bin, frpb);
        if (start == 0.0) start = __dmul_rn (frpb, 0.5);                                   // :320-321
        const double end = __dmul_rn ((double) (bin + 1), frpb);
        const double ra = legacy_ratio (start, r.f0), rb = legacy_ratio (end, r.f0);
        if (floor (ra) != floor (rb)) continue;                                            // :326-327
        const double rr = ra < rb ? ra : rb;
        acc += (rr - floor (rr)) * __ddiv_rn ((double) mg[bin], r.sum);                    // :329-333
    }
    acc = block_sum (acc, red);
    if (t == 0) o[FX_LEGACY_INHARM] = (float) acc;
}

// ---- L6 ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__ (kLegacyThreads) k_legacy_zcr (const LegacyParams p)
{
    __shared__ int wsum[8];
    const int t = threadIdx.x;
    const long row = blockIdx.x;
    const long track = row / p.n_frames;
    const int frame = (int) (row % p.n_frames);
    const float* a = p.audio + track * p.track_stride + (long) frame * p.step;
    int c = 0;
    for (int s = t; s < p.step - 1; s += kLegacyThreads)                                   // :527-535
    {
        const float first = a[s], second = a[s + 1];
        if ((first > 0.0f && __fsub_rn (first, second) > first) || (first < 0.0f && __fsub_rn (first, second) < first)) ++c;
    }
    c = __reduce_add_sync (0xffffffffu, c);
    if ((t & 31) == 0) wsum[t >> 5] = c;
    __syncthreads();
    if (t == 0)
    {
        int tot = 0;
        for (int w = 0; w < kLegacyThreads / 32; ++w) tot += wsum[w];
        p.out[row * FX_LEGACY_NUM + FX_LEGACY_ZCR] = (float) tot * 2.0f / (float) p.step;  // :538
    }
}

} // namespace

} // namespace fx

// ---- C ABI ------------------------------------------------------------------------------------------------------------
extern "C" fx_status fx_legacy_analyse_host (int device, int window, double sample_rate, const float* audio, long track_stride,
                                            long n_samples, int n_tracks, int n_frames, float* out, float* log_attack)
{
    using namespace fx;
    if (! audio || ! out || n_tracks < 1 || n_frames < 1 || n_samples < n_frames || track_stride < n_samples || ! (sample_rate > 0.0))
        return FX_ERR_INVALID_ARG;
    if (window != 1024 && window != 2048 && window != 4096) return FX_ERR_UNSUPPORTED;
    int ndev = 0;
    if (cudaGetDeviceCount (&ndev) != cudaSuccess || ndev == 0) return FX_ERR_NO_DEVICE;          // no CPU fallback
    if (cudaSetDevice (device) != cudaSuccess) return FX_ERR_INVALID_ARG;

    const int N = window, nb = N / 2 + 1, nbp = (nb + 3) & ~3;
    const long rows = (long) n_tracks * n_frames;
    LegacyParams p{};
    float *d_audio = nullptr, *d_mags = nullptr, *d_out = nullptr, *d_la = nullptr;
    double* d_fsum = nullptr; int* d_prev = nullptr; LegacyRec* d_rec = nullptr;
    float2 *d_tw1f = nullptr, *d_tw2 = nullptr;
    cudaStream_t s = nullptr;
    fx_status st = FX_ERR_CUDA;
    std::vector<float2> tw2, tw1f;
    build_twiddles (N, tw2, tw1f);
    double bv = 0.0;                                                                        // :589-593 binVar, the reference's order
    for (double i = 0.0; i < (double) nb; i++) { const double ni = i / (double) nb; bv += (ni - 0.5) * (ni - 0.5); }
    bv /= (double) nb;
#define FXL(call) do { if ((call) != cudaSuccess) goto done; } while (0)
    FXL (cudaStreamCreateWithFlags (&s, cudaStreamNonBlocking));
    FXL (cudaMalloc (&d_audio, (size_t) n_tracks * (size_t) n_samples * sizeof (float)));
    FXL (cudaMalloc (&d_mags, (size_t) rows * nbp * sizeof (float)));
    FXL (cudaMalloc (&d_out, (size_t) rows * FX_LEGACY_NUM * sizeof (float)));
    FXL (cudaMalloc (&d_la, (size_t) n_tracks * sizeof (float)));
    FXL (cudaMalloc (&d_fsum, (size_t) rows * sizeof (double)));
    FXL (cudaMalloc (&d_prev, (size_t) rows * sizeof (int)));
    FXL (cudaMalloc (&d_rec, (size_t) rows * sizeof (LegacyRec)));
    FXL (cudaMalloc (&d_tw1f, tw1f.size() * sizeof (float2)));
    FXL (cudaMalloc (&d_tw2, tw2.size() * sizeof (float2)));
    FXL (cudaMemcpyAsync (d_tw1f, tw1f.data(), tw1f.size() * sizeof (float2), cudaMemcpyHostToDevice, s));
    FXL (cudaMemcpyAsync (d_tw2, tw2.data(), tw2.size() * sizeof (float2), cudaMemcpyHostToDevice, s));
    FXL (cudaMemcpy2DAsync (d_audio, (size_t) n_samples * sizeof (float), audio, (size_t) track_stride * sizeof (float),
                            (size_t) n_samples * sizeof (float), (size_t) n_tracks, cudaMemcpyHostToDevice, s));
    FXL (cudaMemsetAsync (d_out, 0, (size_t) rows * FX_LEGACY_NUM * sizeof (float), s));
    p.audio = d_audio; p.track_stride = n_samples; p.n_samples = n_samples; p.n_frames = n_frames;
    p.step = (int) (n_samples / n_frames);                                                  // :130
    p.nb = nb; p.nbp = nbp; p.sample_rate = sample_rate; p.bin_var = bv;
    p.mags = d_mags; p.fsum = d_fsum; p.prev_idx = d_prev; p.rec = d_rec; p.out = d_out; p.log_attack = d_la;
    p.tw1f = d_tw1f; p.tw2 = d_tw2;
    if (N == 1024)      k_legacy_spectrum<4><<<(unsigned) rows, 64, 0, s>>> (p);
    else if (N == 2048) k_legacy_spectrum<8><<<(unsigned) rows, 128, 0, s>>> (p);
    else                k_legacy_spectrum<16><<<(unsigned) rows, 256, 0, s>>> (p);
    k_legacy_prev<<<(unsigned) ((n_tracks + 127) / 128), 128, 0, s>>> (p, n_tracks);
    k_legacy_features<<<(unsigned) rows, kLegacyThreads, 0, s>>> (p);
    k_legacy_hysteresis<<<(unsigned) ((n_tracks + 127) / 128), 128, 0, s>>> (p, n_tracks);
    k_legacy_inharm<<<(unsigned) rows, kLegacyThreads, 0, s>>> (p);
    k_legacy_zcr<<<(unsigned) rows, kLegacyThreads, 0, s>>> (p);
    FXL (cudaGetLastError());
    FXL (cudaMemcpyAsync (out, d_out, (size_t) rows * FX_LEGACY_NUM * sizeof (float), cudaMemcpyDeviceToHost, s));
    if (log_attack) FXL (cudaMemcpyAsync (log_attack, d_la, (size_t) n_tracks * sizeof (float), cudaMemcpyDeviceToHost, s));
    FXL (cudaStreamSynchronize (s));
    st = FX_OK;
#undef FXL
done:
    cudaFree (d_audio); cudaFree (d_mags); cudaFree (d_out); cudaFree (d_la); cudaFree (d_fsum); cudaFree (d_prev); cudaFree (d_rec);
    cudaFree (d_tw1f); cudaFree (d_tw2);
    if (s) cudaStreamDestroy (s);
    return st;
}

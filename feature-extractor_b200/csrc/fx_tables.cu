// fx_tables.cu -- host-side tables of the analysis kernel: FFT twiddles and the per-lag harmonic / exact-ratio tables,
// all evaluated in the reference's own double arithmetic (citations relative to /root/reference/Source/).
#include "fx_tables.h"
#include <cmath>

namespace fx {

// twiddle tables in the layout fx_fft.cuh expects; evaluated in double, rounded to fp32 (as juce::FFT does)
void build_twiddles (int N, std::vector<float2>& tw2, std::vector<float2>& tw1f)
{
    const int R1 = N / 256;
    const double pi = 3.14159265358979323846;
    // the two factors of a stage-1 twiddle: tw1[(k1 - 1) * 32 + mh] = W_N^(16 mh k1), tw1[(k1 - 1) * 32 + 16 + ml] = W_N^(ml k1)
    std::vector<float2> tw1 ((size_t) (R1 - 1) * 32, make_float2 (1.0f, 0.0f));
    for (int k1 = 1; k1 < R1; ++k1)
        for (int i = 0; i < 16; ++i)
        {
            const double pa = -2.0 * pi * (double) ((long) 16 * i * k1 % N) / (double) N;     // W_N^(16 mh k1)
            const double pb = -2.0 * pi * (double) (i * k1) / (double) N;                      // W_N^(ml k1)
            tw1[(size_t) (k1 - 1) * 32 + i]      = make_float2 ((float) cos (pa), (float) sin (pa));
            tw1[(size_t) (k1 - 1) * 32 + 16 + i] = make_float2 ((float) cos (pb), (float) sin (pb));
        }
    // the full stage-1 table: W_N^(m k1) = W_N^(16 mh k1) * W_N^(ml k1), m = 16 mh + ml, as the fp32 product of the two
    // factors above with the roundings of the kernel's former in-line product (one rounded product, one FMA per part)
    tw1f.assign ((size_t) (R1 - 1) * 256, make_float2 (1.0f, 0.0f));
    for (int k1 = 1; k1 < R1; ++k1)
        for (int m = 0; m < 256; ++m)
        {
            const float2 wa = tw1[(size_t) (k1 - 1) * 32 + (m >> 4)], wb = tw1[(size_t) (k1 - 1) * 32 + 16 + (m & 15)];
            volatile float pyy = wa.y * wb.y, pxy = wa.x * wb.y;
            tw1f[(size_t) (k1 - 1) * 256 + m] = make_float2 (fmaf (wa.x, wb.x, -pyy), fmaf (wa.y, wb.x, pxy));
        }
    tw2.assign (15 * 16, make_float2 (1.0f, 0.0f));
    for (int k2 = 1; k2 < 16; ++k2)
        for (int n3 = 0; n3 < 16; ++n3)
        {
            const double ph = -2.0 * pi * (double) (n3 * k2) / 256.0;
            tw2[(size_t) (k2 - 1) * 16 + n3] = make_float2 ((float) cos (ph), (float) sin (ph));
        }
}

// f0 and the harmonic bins as functions of the integer lag, in the reference's arithmetic (see AnalyseParams)
void build_lag_tables (int N, double sample_rate, std::vector<short>& her_tab)
{
    const int M = N / 2;
    const double nyquist = sample_rate / 2.0;
    const double frpb = nyquist / (double) M;                       // HarmonicCharacteristics.h:53
    her_tab.assign ((size_t) (N + 1) * FX_HER_TAB_STRIDE, (short) -1);
    auto clamp_short = [] (double v) { return (short) (v > 32767.0 ? 32767.0 : (v < -32768.0 ? -32768.0 : v)); };
    for (int slot = 0; slot <= N; ++slot)
    {
        const double lag = slot == 0 ? -1.0 : (double) slot;
        const double f0 = (nyquist * 2.0) / lag;                    // PitchAnalyser.h:57
        short* row = her_tab.data() + (size_t) slot * FX_HER_TAB_STRIDE;
        const double f0_bin_d = floor (f0 / frpb);                  // :246-249
        row[18] = clamp_short (f0_bin_d);
        const int f0_bin = (int) f0_bin_d;
        for (int l = 0; l < 15; ++l)
        {
            const double fr = f0 * ldexp (1.0, -(l + 1));           // f0 / 2^(l+1), exact scaling (:160-161)
            const double hb = floor (fr / frpb);
            // a sub-octave landing in f0's own bin is skipped (:163-164)
            if (hb >= 0.0 && hb < (double) M && (int) hb != f0_bin) row[l] = (short) hb;
        }
        for (int h = 1; h <= 3; ++h)
        {
            const double fr = f0 * (double) h;                      // :171-172
            const double hb = floor (fr / frpb);
            // harmonics stop at the first bin >= M (:174-175); they ascend, so skipping every bin >= M is the same
            if (hb >= 0.0 && hb < (double) M) row[14 + h] = (short) hb;
        }
    }
}

// Inharmonicity fractions for the (lag, bin) pairs whose edge ratios may be exact integers -- there the reference's own fp64
// rounding decides on which side of the integer a ratio lands, so the value is taken from the reference's arithmetic, evaluated
// here (HarmonicCharacteristics.h:223-236, :251-259), instead of being derived on the GPU.  Layout per lag (step = N / gcd (lag, N)):
//   [ex_off[lag] + 2 q]     bin = q step      (start edge: bin lag is a multiple of N)
//   [ex_off[lag] + 2 q + 1] bin = q step - 1  (end edge: (bin + 1) lag is a multiple of N),   q = 0 .. M / step
// and, for lag = 2^b only, 2 * 13 entries in front of them for the bins below f0's:
//   [ex_off[lag] - 26 + 2 a] bin = 2^a,  [ex_off[lag] - 26 + 2 a + 1] bin = 2^a - 1   (bin lag or (bin + 1) lag divides N)
void build_exact_ratio_table (int N, double sample_rate, std::vector<double>& ex_tab, std::vector<int>& ex_off)
{
    const int M = N / 2;
    const double nyquist = sample_rate / 2.0;
    const double frpb = nyquist / (double) M;
    auto ratio = [] (double f1, double f2)                         // getFrequencyRatio (:251-259)
    {
        if (f1 == f2) return 1.0;
        const double higher = f1 > f2 ? f1 : f2;
        const double lower = higher == f1 ? f2 : f1;
        return higher / lower;
    };
    auto fraction = [&] (int bin, double f0)                       // :223-236
    {
        if (bin < 0 || bin >= M) return 0.0;
        double start = (double) bin * frpb;
        if (start == 0.0) start = frpb * 0.5;
        const double end = (double) (bin + 1) * frpb;
        const double ra = ratio (start, f0), rb = ratio (end, f0);
        if (floor (ra) != floor (rb)) return 0.0;
        const double r = ra < rb ? ra : rb;
        return r - floor (r);
    };
    ex_tab.clear();
    ex_off.assign ((size_t) N + 1, 0);
    for (int lag = 1; lag <= N; ++lag)
    {
        const double f0 = (nyquist * 2.0) / (double) lag;           // PitchAnalyser.h:57
        const int g = lag & -lag, step = N / g;
        if ((lag & (lag - 1)) == 0)
            for (int a = 0; a < 13; ++a)
            {
                ex_tab.push_back (fraction (1 << a, f0));
                ex_tab.push_back (fraction ((1 << a) - 1, f0));
            }
        ex_off[(size_t) lag] = (int) ex_tab.size();
        for (int q = 0; q <= M / step; ++q)
        {
            ex_tab.push_back (fraction (q * step, f0));
            ex_tab.push_back (fraction (q * step - 1, f0));
        }
    }
}

} // namespace fx

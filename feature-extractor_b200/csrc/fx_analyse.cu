// fx_analyse.cu -- K1, the per-frame analysis kernel (sm_100a), and K1b, the per-frame finalisation.
//
// One CTA walks a chunk of consecutive frames of one track.  Per frame it reproduces, on the GPU, the two
// analyser bodies of the reference (all citations relative to /root/reference/Source/):
//   RealTimeSpectralAnalyser::run  (RealTimeAnalyser.h:205-229)   RMS, Bartlett window, FFT, spectral features, slope
//   RealTimeHarmonicAnalyser::run  (RealTimeAnalyser.h:145-172)   RMS, one-pole filter, window, 2 FFTs, pitch, harmonic features
// including their quirks (SURVEY.md section 8a): "magnitude" = Re(X)^2, asymmetric Bartlett window, harmonic
// features on the un-windowed frame, integer pitch lag, raw fp64 flatness product with IEEE under/overflow,
// previous spectrum not updated on silent frames.
//
// Data movement: the hop's new samples arrive as 16-byte asynchronous copies (cp.async / LDGSTS, completion handed to an
// mbarrier) in a SKEWED shared-memory ring holding the N-sample window, so each input sample crosses HBM once per chunk and
// the float4 reads of the filter pass are bank-conflict free; the next hop is prefetched as soon as the frame's last read of
// the ring is behind a barrier and lands during the pitch / harmonic passes.  K1b streams K1's records through shared
// memory with cp.async.bulk (the TMA bulk copy).
// The reference runs four real-input transforms per hop; here they are packed into TWO complex FFTs, both through
// ONE out-of-line copy of the FFT code (the kernel is instruction-cache bound otherwise):
//   FFT-alpha  z = x w + i onepole (x) w   -> B = FFT (x w): Re B (+ Im B for the slope quirk), C: P[k] = Re C[k]^2,
//              separated by conjugate symmetry for each thread's own 8 consecutive bins
//   FFT-beta   z = x + i 2^k P             -> Re Z = Re A (raw frame, harmonic features); Im Z[s] + Im Z[N-s] = 2^(k+1) D[s],
//              D = FFT (P) real and even = N x the real part of the inverse transform the reference performs
//              (PitchAnalyser.h:120), which is all that can reach the lag search (PitchAnalyser.h:163)
// K1 leaves the per-frame sums in a FrameRec; K1b (one thread per frame) applies the scalar tail of the
// reference (pow / log10 / sqrt, clamps, gates) so that no serial libm code sits inside the frame loop.
// Every sum accumulates in fp64 per thread like the reference, and across the warps; across the 32 lanes of a warp the raw
// moments that K1b subtracts from each other stay fp64, the other partials (sums of positive terms) are added in fp32.
// No tensor cores: nothing here is a GEMM.
#include "fx_fft.cuh"
#include "fx_kernels.cuh"
#include <math.h>

// The spectral features take ONE pass over a thread's bins.  Spread, slope and energy variance are moments about values
// (centroid, mean energy, largest magnitude) that are only known after a block reduction; expanded, they are combinations
// of raw moments that the first pass can accumulate:  with x = (bin + 1/2) / M, S0 = sum mag, W1 = sum x mag,
// S2 = sum x^2 mag, S4 = sum mag^2
//     sum (x - c)^2 mag        = S2 - 2 c W1 + c^2 S0                       (SpectralCharacteristics.h:135-139)
//     sum bin * mag / maxE     = (M W1 - S0 / 2) / maxE                     (:175)
//     sum (mag / maxE - mean)^2 = S4 / maxE^2 - M mean^2                    (:182-190)
// in fp64 (the cancellation costs a few of its 16 digits on features compared at 1e-4).  K1b forms them.
//
// Every optimisation in this file was A/B-timed on a B200 against the form it replaced (DESIGN.md section 7,
// profiles/r02_v2*_ab_*.txt); the losing forms are gone.  Three are selected per window size (kPackFilter, kFluxF32Cmp,
// kLhrRange in k_analyse): at N = 4096 the kernel sits at its 80-register budget and what trims instructions elsewhere makes
// ptxas spill there.  Dropped after measurement: a MUFU-approximate flatness eps, packed arithmetic in the split, fp32
// cross-warp sums of rms / magnitude / harmonic sums (spills), a per-warp queue dealing the peaks out one per lane (+1 .. 3 %).

namespace fx {

// ---------------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + bulk async copy (TMA, non-tensor form)
__device__ __forceinline__ uint32_t smem_u32 (const void* p) { return (uint32_t) __cvta_generic_to_shared (p); }

__device__ __forceinline__ void mbar_init (uint64_t* bar, uint32_t count)
{
    asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32 (bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx (uint64_t* bar, uint32_t bytes)
{
    asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32 (bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive (uint64_t* bar)
{
    asm volatile ("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32 (bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait (uint64_t* bar, uint32_t parity)
{
    asm volatile (
        "{\n"
        ".reg .pred p;\n"
        "FX_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra FX_WAIT_DONE;\n"
        "bra FX_WAIT_LOOP;\n"
        "FX_WAIT_DONE:\n"
        "}\n" :: "r"(smem_u32 (bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s (void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                  :: "r"(smem_u32 (dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32 (bar)) : "memory");
}
// 16-byte asynchronous copy global -> shared (LDGSTS: no register staging) and the arrival of a thread's copies at an mbarrier
__device__ __forceinline__ void cp_async16 (void* dst_smem, const void* src_gmem)
{
    asm volatile ("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32 (dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_arrive (uint64_t* bar)       // arrives (without raising the expected count) once this thread's copies have landed
{
    asm volatile ("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" :: "r"(smem_u32 (bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile ("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------------
// small numeric helpers.  Margins are diagnostics: fp32 with the fast reciprocal is plenty.
__device__ __forceinline__ float relmargin_f (float a, float b)
{
    const float m = fmaxf (fabsf (a), fabsf (b));
    return (m > 0.0f) ? __fdividef (fabsf (a - b), m) : 0.0f;
}
__device__ __forceinline__ float relmargin_d (double a, double b)
{
    const float m = (float) fmax (fabs (a), fabs (b));
    return (m > 0.0f) ? __fdividef ((float) fabs (a - b), m) : 0.0f;
}
// margin of a comparison between cnd values with fp32 uncertainties ua, ub (the CPU checker computes the same margin in its pitch estimator)
__device__ __forceinline__ float noisy_margin (float a, float ua, float b, float ub)
{
    const float gap = fabsf (a - b) - (ua + ub);
    const float m = fmaxf (fabsf (a), fabsf (b));
    return (gap > 0.0f && m > 0.0f) ? __fdividef (gap, m) : 0.0f;
}

// fp32 uncertainty of cnd[s] = d^2 s / sum when d carries an absolute error e_abs: (2 |d| e + e^2) s / sum = c r (2 + r),
// r = e / |d|.  d == 0 means the value is pure rounding noise.
__device__ __forceinline__ float cnd_uncertainty (float c, float d, float e_abs)
{
    const float ad = fabsf (d);
    if (! (ad > 0.0f)) return 1.0e30f;
    const float r = __fdividef (e_abs, ad);
    return c * r * (2.0f + r);
}

// Conservative (never over-estimating) relative gap between two non-negative fp32 values from the distance of
// their bit patterns: |a - b| / max (a, b) >= ulps * 2^-24.  Three integer instructions per comparison.
__device__ __forceinline__ unsigned ulp_gap (float a, float b)
{
    const int d = (int) __float_as_uint (a) - (int) __float_as_uint (b);
    return (unsigned) (d < 0 ? -d : d);
}
__device__ __forceinline__ float ulps_to_margin (unsigned u)
{
    return u >= (1u << 24) ? 1.0f : (float) u * (1.0f / 16777216.0f);
}
__device__ __forceinline__ float rcp_approx (float x)
{
    float r;
    asm ("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// floor (NN / d) for 1 <= d <= NN <= 4096 from an approximate fp32 reciprocal r of d (relative error a few 2^-23: the estimate is
// off by at most one, and one comparison settles it).
template <int NN> __device__ __forceinline__ int idiv_n (int d, float r)
{
    int q = __float2int_rz ((float) NN * r);
    q += ((q + 1) * d <= NN) ? 1 : 0;
    q -= (q * d > NN) ? 1 : 0;
    return q;
}
__device__ __forceinline__ double ldexp_normal (double m, int e)       // m in [0.5, 1), result a normal double
{
    return (m * 2.0) * __hiloint2double ((e - 1 + 1023) << 20, 0);
}

// extended-range product of fp64 magnitudes: value = m * 2^e with m in [0.5, 1).  Inputs are squares of fp32
// values, i.e. normal doubles, so the exponent field can be read directly.
struct ME { double m; int e; };
__device__ __forceinline__ ME me_one() { ME r; r.m = 0.5; r.e = 1; return r; }
__device__ __forceinline__ ME me_from (double x)
{
    ME r;
    const int hi = __double2hiint (x);
    r.e = ((hi >> 20) & 0x7ff) - 1022;
    r.m = __hiloint2double ((hi & 0x800fffff) | 0x3fe00000, __double2loint (x));
    return r;
}
__device__ __forceinline__ ME me_mul (ME a, ME b)
{
    ME r;
    r.m = a.m * b.m;                     // in [0.25, 1)
    r.e = a.e + b.e;
    if (r.m < 0.5) { r.m *= 2.0; r.e -= 1; }
    return r;
}

// Sum K (a power of two <= 8) doubles over the warp with a transposed butterfly: each of the first log2 K steps halves the
// number of values a lane carries (it keeps one half of the pairs and sends the other half to its partner), the remaining
// steps are plain butterflies on one value: K - 1 + (5 - log2 K) exchanges instead of 5 K.  Afterwards v[0] of every lane
// holds the warp total of value warp_sum_slot<K> (lane).
template <int K> __device__ __forceinline__ int warp_sum_slot (int lane)
{
    int idx = 0;
    #pragma unroll
    for (int b = 0; (K >> (b + 1)) > 0; ++b) idx += ((lane >> b) & 1) * (K >> (b + 1));
    return idx;
}
template <int K, typename V> __device__ __forceinline__ void warp_sum_t (V (&v)[K], int lane)
{
    int b = 0;
    #pragma unroll
    for (int half = K / 2; half > 0; half >>= 1, ++b)
    {
        const bool up = (lane >> b) & 1;
        #pragma unroll
        for (int i = 0; i < half; ++i)
        {
            const V keep = up ? v[i + half] : v[i];
            const V send = up ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync (0xffffffffu, send, 1 << b);
        }
    }
    #pragma unroll
    for (int off = K; off < 32; off <<= 1) v[0] += __shfl_xor_sync (0xffffffffu, v[0], off);
}
__device__ __forceinline__ float warp_sumf (float v)
{
    #pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync (0xffffffffu, v, off);
    return v;
}
// Single-instruction warp reductions (REDUX) on integers; non-negative floats order like their bit patterns, so the
// maxima of |Re| and the minima of the (non-negative) margins go through the same instruction.
__device__ __forceinline__ unsigned warp_minu (unsigned v) { return __reduce_min_sync (0xffffffffu, v); }
__device__ __forceinline__ int warp_addi (int v) { return __reduce_add_sync (0xffffffffu, v); }
__device__ __forceinline__ float warp_max_nonneg (float v) { return __uint_as_float (__reduce_max_sync (0xffffffffu, __float_as_uint (v))); }
__device__ __forceinline__ float warp_min_nonneg (float v) { return __uint_as_float (__reduce_min_sync (0xffffffffu, __float_as_uint (v))); }

// ---------------------------------------------------------------------------------------------------------
template <int R1> struct Smem
{
    using D = FftDims<R1>;
    static constexpr int N = D::N, M = N / 2, T = D::T, NW = T / 32;

    float2   ex[D::EX_LEN];          // FFT exchange buffer; doubles as two fp32 work arrays (skewed, N*17/16 floats each)
    // The sample ring and the P / Re A array are SKEWED by one float4 per 32 floats (sk32 below): a thread reads 16 (8)
    // consecutive floats as float4s, i.e. the lanes of a quarter warp are 64 (32) bytes apart and would share two (four) of the
    // eight 16-byte bank groups; with the skew every quarter warp covers all eight.  Runs of 32 consecutive floats that start at
    // a multiple of 32 stay contiguous (the gather of FFT-beta, the 128-byte pieces of the bulk copies).
    alignas (128) float ring[N + N / 8];       // ring[sk32 (a & (N-1))] = absolute sample a of the track (bulk-copy destination, float4 reads)
    alignas (16) float pa[M + M / 8 + 4];      // pa[sk32 (k)]: P[k] = Re C[k]^2, k = 0..M (input of FFT-beta), then Re A[k] (harmonic features)
    // Per-warp partials every thread reads back after a barrier.  What one reader needs of a warp sits in ONE 16-byte slot: a
    // broadcast LDS.128 per warp instead of one load per value (these reads were ~40 of the 230 LDS per thread and frame).
    struct alignas (16) P1Slot  { double s0; float maxre; float psum; };      // pass 1: magnitude sum, largest |Re|, sum of P^2
    struct alignas (16) ScanSlot { double m; int e; float mf; };              // flatness product scan, warp totals (the prefix reads e and mf = (float) m)
    struct alignas (16) LagSlot { float hsum, hmax; unsigned first_cross, best; };      // harmonic magnitude sum, largest |Re A|; first lag under the threshold, smallest cnd (bit pattern)
    alignas (16) double rms[NW];     // sum of squares of the frame, warp totals
    P1Slot   p1s[NW];
    ScanSlot scan[NW];
    alignas (16) float pscan[NW];    // pitch cumulative sum scan, warp totals
    LagSlot  lags[NW];
    unsigned ugidx[NW];             // first index holding the smallest cnd (only formed when no lag crosses the threshold)
    unsigned ucodes[NW];            // flatness product: earliest range-event thread of the warp
    float    fmins[2][NW];           // [0] flatness gate margin, [1] peak margin (diagnostics)
    float    pmins[2][NW];           // pitch margin / runner-up partials
    union
    {
        unsigned short ndm[T];       // per 16-lag segment: bit j set when cnd[j + 1] < cnd[j] does NOT hold (PitchAnalyser.h:178); dead after the lag derivation
        double   ev_chunk[32];       // 32 gated magnitudes of the product's continuation (record stage, behind the frame's last barrier)
    };
    double   ev_prod[NW];           // flatness product replayed by the warp's earliest range event
    float    d0;                     // autocorrelation at lag 0 (noise floor of the pitch margin)
    uint64_t mbar;
    const float2* tw1f;
};

extern __shared__ __align__ (128) unsigned char fx_smem_raw[];

// position of element i of an array skewed by one float4 per 32 floats
__device__ __forceinline__ int sk32 (int i) { return i + ((i >> 5) << 2); }

struct V16 { float2 v[16]; };

// The one copy of the FFT: stage 1 (+ twiddle) -> block barrier -> stage 2 (+ twiddle) -> warp barrier -> stage 3, every
// stage in place.  v: slot q * R1 + n1 = input n1 of stage-1 butterfly m0 + T q.  The spectrum is left in the exchange
// buffer at zpos (k); the caller puts a block barrier between this call and the first read of another thread's bins, and
// guarantees that nobody still reads the buffer on entry (other than this thread's own stage-1 inputs).
template <int R1>
__device__ __noinline__ void fft_core (V16 io, int m0)
{
    Smem<R1>& sm = *reinterpret_cast<Smem<R1>*> (fx_smem_raw);
    const int t = threadIdx.x;
    fft_stage1_store<R1, false> (io.v, m0, sm.ex, sm.tw1f);
    __syncthreads();
    fft_stage2<R1, false, true> (t, sm.ex, reinterpret_cast<const float2*> (sm.ring + 32));
    __syncwarp();                                           // rows are private to a half warp from here on
    fft_stage3<R1, false> (t, sm.ex);
}
// fft_core_pruned: the same transform for the parity-mode kernels, which call it for both transforms.  even (uniform): the input
// is even and only the rows k1 <= R1 / 2 of the spectrum are computed (fx_fft.cuh); X[k] of the other rows is X[N - k], in a
// computed row.  The half warps of the skipped rows leave after the block barrier; the row boundary splits a warp at every
// window size, so the warp barriers name the row's half warp only.  A runtime flag rather than a second out-of-line copy:
// with two copies in one kernel ptxas spills 24 bytes at N = 4096.
template <int R1>
__device__ __noinline__ void fft_core_pruned (V16 io, int m0, bool even)
{
    Smem<R1>& sm = *reinterpret_cast<Smem<R1>*> (fx_smem_raw);
    const int t = threadIdx.x;
    fft_stage1_store<R1, false, true> (io.v, m0, sm.ex, sm.tw1f, even);
    __syncthreads();
    if (even && (t >> 4) > R1 / 2) return;
    const unsigned rowmask = 0xffffu << (t & 16);
    fft_stage2<R1, false, true> (t, sm.ex, reinterpret_cast<const float2*> (sm.ring + 32));
    __syncwarp (rowmask);                                   // rows are private to a half warp from here on
    fft_stage3<R1, false> (t, sm.ex, rowmask);
}

// MG: also compute the decision margins (diagnostics, FX_DIAG_*_MARGIN).  They feed nothing: a call that does not ask for the
// diagnostics runs the instantiation without them -- same features, bit for bit (tests/test_gpu_parity.py).
// Resident CTAs per SM the kernel is compiled for (register budget = 65536 / (threads x CTAs)): 3 x 256 threads at 80 registers
// (N = 4096: a fourth CTA would need 64 registers AND 8 KB less shared memory); 7 x 128 and 13 x 64 threads at 72 registers
// (N = 2048 / 1024: 28 / 26 warps per SM instead of 24; the seventh / thirteenth CTA fits the shared memory only with the compact
// stage-2 twiddle table, 512 B instead of 1920 B).  Measured against 6 / 12 CTAs at 80 registers: 32.45 vs 32.78 ms at N = 2048,
// 33.82 vs 33.98 ms at N = 1024 (profiles/r02_v23_ab_occupancy.txt).
constexpr int kCtasR16 = 3, kCtasR8 = 7, kCtasR4 = 13;
// (233 472 bytes of shared memory per SM, 1 KB of it reserved per resident CTA)
static_assert (kCtasR16 * (sizeof (Smem<16>) + 1024) <= 233472, "three CTAs of N = 4096 per SM");
static_assert (kCtasR8 * (sizeof (Smem<8>) + 1024) <= 233472, "resident CTAs of N = 2048 per SM");
static_assert (kCtasR4 * (sizeof (Smem<4>) + 1024) <= 233472, "resident CTAs of N = 1024 per SM");
// SP: power-spectrum mode (FX_SPECTRUM_POWER).  Each of the three spectra is handed on as (|X[k]|, 0) instead of
// (Re X[k], Im X[k]): |B| to the spectral passes and the previous spectrum, P = |C|^2 to FFT-beta, |A| to the harmonic
// pass.  Everything downstream squares or compares these values exactly as it squares and compares Re, so the two
// places that form them (the split after FFT-alpha, the hand-over of A after FFT-beta) are the only branches on SP;
// the instantiations without it are the parity mode, unchanged.
// SO: the spectrum export (fx_analyse_device_spectrum).  Each frame's mag[m] = cr[m]^2, the per-bin energy the spectral pass
// reads, is also stored to p.spec; the instantiations without it compile to the same instructions as before SO existed.
template <int R1, bool MG, bool SP, bool SO>
__global__ void __launch_bounds__ (16 * R1, (R1 == 16 ? kCtasR16 : (R1 == 8 ? kCtasR8 : kCtasR4)))
k_analyse (const AnalyseParams p)
{
    using D = FftDims<R1>;
    using S = Smem<R1>;
    constexpr int N = D::N, M = N / 2, T = D::T, NW = T / 32, Q1 = D::Q1;
    constexpr int LOG_N = R1 == 16 ? 12 : (R1 == 8 ? 11 : 10);
    // The record stage's parts run on the CTA's last warps: the upper bins have fewer peaks, so those warps leave the peak
    // loop first (which of the three takes which part is immaterial: profiles/r02_v29c_ab_role_permutations_4096.txt)
    constexpr int kRoleHer  = NW - 1;
    constexpr int kRoleHead = NW >= 2 ? NW - 2 : 0;
    constexpr int kRoleFlat = NW >= 3 ? NW - 3 : 0;
    // Per window size (profiles/r02_v28a_ab_*.txt): the filter pass on packed f32x2 instructions (two samples per instruction,
    // IEEE per half: the same values) pays 1.2 - 1.4 % at N = 2048 / 1024 (no spills there) and costs 2.7 % at N = 4096
    // (80-register budget: 40 bytes of spills).  Its three parts -- sums of squares, the (x gain, x c1 gain) multiply, decay +
    // ramp -- were also timed alone at N = 4096: 0 / +0.1 / +2.1 % (profiles/r02_v29a_ab_4096.txt).
    constexpr bool kPackFilter = R1 <= 8;
    // Per window size (profiles/r02_v26a_ab_*.txt, r02_v28a_ab_*.txt): "magnitude rose" decided on |Re| with a predicated add
    // instead of selects on the fp64 difference trims instructions where they fit and spills at N = 4096 (+0.6 % there).
    constexpr bool kFluxF32Cmp = R1 <= 8;
    // Per window size (profiles/r02_v28b_ab_*.txt): the low-energy sum as the magnitude sum of the threads below the boundary
    // bin, only the thread that straddles it testing bins, pays at N >= 2048 and costs 0.8 % at N = 1024 (spills).
    constexpr bool kLhrRange = R1 >= 8;
    // Per window size (profiles/r02_v35_even_beta_ab.txt): FFT-beta on the even part of the frame with the mirror rows of the
    // spectrum skipped (parity mode only: the power mode reads Im A) pays 3.6 % at N = 4096 (80 registers, no spills).  At
    // N = 2048 it pays 1.4 % but makes ptxas spill 8 bytes; at N = 1024 (one skipped row of four, 8 bytes of spills) it costs 3.0 %.
    constexpr bool kEvenBeta = ! SP && R1 == 16;

    S& sm = *reinterpret_cast<S*> (fx_smem_raw);
    float* workf = reinterpret_cast<float*> (sm.ex);          // fp32 view, skewed index phys (n)
    float* workg = workf + D::EX_LEN;                          // second fp32 array in the same buffer

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const long cta = blockIdx.x;
    const int chunk = (int) (cta % p.n_chunks);
    const long track = cta / p.n_chunks;
    const int f_begin = chunk * p.frames_per_chunk;
    const int f_end = min (p.n_frames, f_begin + p.frames_per_chunk);
    if (f_begin >= f_end)
    {
        if (t == 0) p.first_idx[track * p.n_chunks + chunk] = -1;
        return;
    }

    const int H = p.hop, NB = N >> p.log2_hop;
    const float gain = p.gain[track];
    const float* src = p.audio + track * p.track_stride;
    const float* tail = p.tail_in + track * (long) (N - H);

    // The stage-2 twiddles by powers (fx_fft.cuh), rows k2 = 1, 2, 4, 8, live in the ring's holes.  At N = 2048 / 1024 they
    // cost ~1 % by themselves and buy the shared memory for one more resident CTA: 512 B instead of the full table's 1920 B.
    static_assert (4 * 16 / 2 <= N / 32, "one hole per two stage-2 twiddles");
    for (int i = t; i < 4 * 16; i += T)
        reinterpret_cast<float2*> (sm.ring + 32)[18 * (i >> 1) + (i & 1)] = p.tw2[((1 << (i >> 4)) - 1) * 16 + (i & 15)];
    if (t == 0) { mbar_init (&sm.mbar, T); sm.tw1f = p.tw1f; }             // every thread arrives once per hop block (its copies, or its stores)
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // ---- fill the ring with the window of the chunk's first frame ------------------------------------
    // frame f (call-relative) ends with hop block f of this call = absolute hop first_hop + f
    {
        const long j_new = p.first_hop + f_begin;
        for (int b = 0; b < NB; ++b)
        {
            const long j = j_new - (NB - 1) + b;                 // absolute hop index
            const int base = (int) ((j * H) & (N - 1));
            const float* g = nullptr;
            if (j >= p.first_hop)                  g = src + (j - p.first_hop) * H;
            else if (j >= 0)                       g = tail + (j - (p.first_hop - (NB - 1))) * H;
            if (g == nullptr)      { _Pragma ("unroll 1") for (int i = t; i < H; i += T) sm.ring[sk32 (base + i)] = 0.0f; }      // before the stream started (RealTimeAudioAnalysis.h:202)
            else if (! p.use_bulk) { _Pragma ("unroll 1") for (int i = t; i < H; i += T) sm.ring[sk32 (base + i)] = g[i]; }
            else                   { _Pragma ("unroll 1") for (int k = 4 * t; k < H; k += 4 * T) cp_async16 (&sm.ring[sk32 (base + k)], g + k); }
        }
        cp_async_arrive (&sm.mbar);
        __syncthreads();
    }

    uint32_t phase = 0;
    // the chunk's running "previousBinMagnitudes" (as Re values): written after every non-silent frame, re-read by the
    // same thread for the next frame's flux, and left behind for K2 as the chunk's last non-silent spectrum
    float* prev_g = p.last_spec + (track * p.n_chunks + chunk) * (long) M;
    bool have_prev = false;           // false until the chunk's first non-silent frame (its flux is fixed up by K2)
    int first_nonsilent = -1;
    const int lower_portion = M / 5;                                // SpectralCharacteristics.h:65
    const int b0 = 8 * t;                                           // this thread's 8 consecutive bins
    const int pb0 = sk32 (b0);                                      // ... and where they start in the skewed P / Re A array
    const double inv_m = 1.0 / (double) M;                          // exact: M is a power of two
    // where this thread's runs of the spectrum live in the exchange buffer (fx_fft.cuh: zpos): its 8 bins b0 + j and their
    // mirrors N - b0 - j (j = 0 pairs with (N - b0) & (N - 1), j >= 1 with the run that starts at N - b0 - 8), and its 16 lags
    const int zb_own = zpos<R1> (b0), zb_self = zpos<R1> ((N - b0) & (N - 1)), zb_mirror = zpos<R1> (N - b0 - 8);
    const int zl_own = zpos<R1> (16 * t), zl_self = zpos<R1> ((N - 16 * t) & (N - 1)), zl_mirror = zpos<R1> (N - 16 * t - 16);
    // the same ramp over this thread's 16 consecutive samples (filter / pitch layout): w = wseg_0 + j wseg_d
    // The ramp is stored halved: FFT-alpha then delivers Z / 2 (a power-of-two scale commutes with every rounding of the
    // transform), and the split B = (Z[k] + conj Z[N-k]) / 2 needs no multiplications.
    const float wseg_0 = 0.5f * ((16 * t < M) ? (float) (16 * t) * (2.0f / N) : 1.0f - (float) (16 * t - M) * (2.0f / N));
    const float wseg_d = (16 * t < M) ? (1.0f / N) : -(1.0f / N);

    #pragma unroll 1
    for (int f = f_begin; f < f_end; ++f)
    {
        const long j_new = p.first_hop + f;
        const long a0 = (j_new - (NB - 1)) * (long) H;              // absolute sample index of window sample 0
        unsigned char* rec_bytes = p.rec + (size_t) (track * p.n_frames + f) * frame_rec_bytes (N);
        FrameHead* rec = reinterpret_cast<FrameHead*> (rec_bytes);
        WarpPart* rec_w = reinterpret_cast<WarpPart*> (rec_bytes + sizeof (FrameHead));           // [NW]

        mbar_wait (&sm.mbar, phase);
        phase ^= 1u;

        // =========================== one-pole filter + window -> work array ============================
        // AudioFilter::filterAudio (RealTimeAudioAnalysis.h:106-125): y[0] = x[0]; y[n] = (pi/2) x[n] + e^(-pi/2) y[n-1].
        // Each thread owns 16 consecutive samples: it runs the recurrence from a zero state over them, takes the state
        // entering its segment from its left neighbour's zero-state end value (what that misses is e^(-pi/2)^16 = 1.2e-11
        // of the state, far below fp32 resolution) and adds its decaying contribution e^(-pi/2)^(j+1) y_in.  FMAs and
        // the folded gain differ from the reference's separate roundings by an ulp, well inside the rounding of the FFT
        // this feeds.  The work array is free: the previous frame ended with a barrier.  The same pass over the raw
        // samples takes the sum of squares for the RMS (getRMSLevel: fp32 squares, fp64 sum; here 16 squares are summed in
        // fp32 first, 1e-7 relative on a feature compared at 1e-4).
        {
            const int n0 = 16 * t;
            const int r0 = sk32 ((int) ((a0 + n0) & (N - 1)));                                    // 16 consecutive samples stay inside a 32-float group
            const float c1 = p.iir_c1, c2 = p.iir_c2, c1g = __fmul_rn (c1, gain);
            float xs[16], ys[16], xg[16], y;
            float sq0 = 0.0f, sq1 = 0.0f;
            float2 sqp = make_float2 (0.0f, 0.0f);
            #pragma unroll
            for (int q = 0; q < 4; ++q)
            {
                const float4 x4 = *reinterpret_cast<const float4*> (&sm.ring[r0 + 4 * q]);
                xs[4 * q] = x4.x; xs[4 * q + 1] = x4.y; xs[4 * q + 2] = x4.z; xs[4 * q + 3] = x4.w;
                if (kPackFilter)
                {
                    sqp = f2fma (make_float2 (x4.x, x4.y), make_float2 (x4.x, x4.y), sqp); sqp = f2fma (make_float2 (x4.z, x4.w), make_float2 (x4.z, x4.w), sqp);
                }
                else
                {
                    sq0 = fmaf (x4.x, x4.x, sq0); sq1 = fmaf (x4.y, x4.y, sq1); sq0 = fmaf (x4.z, x4.z, sq0); sq1 = fmaf (x4.w, x4.w, sq1);
                }
            }
            if (kPackFilter)
            {
                sq0 = sqp.x; sq1 = sqp.y;
            }
            {
                const float wsq = warp_sumf (sq0 + sq1);
                if (lane == 0) sm.rms[warp] = (double) wsq * ((double) gain * (double) gain);      // AudioDataCollector.h:88 applies the gain
            }
            if (kPackFilter)
            {
                // (x gain, x c1 gain) of a sample in one packed multiply: the first half is the windowed path's sample, the second the filter's input
                #pragma unroll
                for (int j = 0; j < 16; ++j)
                {
                    const float2 r = f2mul (make_float2 (xs[j], xs[j]), make_float2 (gain, c1g));
                    xg[j] = r.x; ys[j] = r.y;
                }
                y = (t == 0) ? xg[0] : ys[0];                                                         // y[0] = x[0]
                ys[0] = y;
                #pragma unroll
                for (int j = 1; j < 16; ++j) { y = fmaf (c2, y, ys[j]); ys[j] = y; }
            }
            else
            {
                y = (t == 0) ? __fmul_rn (xs[0], gain) : __fmul_rn (xs[0], c1g);                     // y[0] = x[0]
                ys[0] = y;
                #pragma unroll
                for (int j = 1; j < 16; ++j) { y = fmaf (c2, y, __fmul_rn (xs[j], c1g)); ys[j] = y; }
            }
            // every lane runs the warm-up of its WARP's first segment from broadcast loads (one wavefront each): an independent
            // chain the scheduler can interleave with the recurrence above, instead of a divergent tail behind it
            float ywarm = 0.0f;
            {
                const int rpw = sk32 ((int) ((a0 + 16 * (t & ~31) - 12) & (N - 1)));
                #pragma unroll
                for (int q = 0; q < 3; ++q)
                {
                    const float4 x4 = *reinterpret_cast<const float4*> (&sm.ring[rpw + 4 * q]);
                    ywarm = fmaf (c2, ywarm, __fmul_rn (x4.x, c1g)); ywarm = fmaf (c2, ywarm, __fmul_rn (x4.y, c1g));
                    ywarm = fmaf (c2, ywarm, __fmul_rn (x4.z, c1g)); ywarm = fmaf (c2, ywarm, __fmul_rn (x4.w, c1g));
                }
            }
            float yin = __shfl_up_sync (0xffffffffu, y, 1);
            if (lane == 0) yin = (t != 0) ? ywarm : 0.0f;
            // e^(-pi/2 (j+1)): the filter constant is fixed by AudioFilter::m = 2 (RealTimeAudioAnalysis.h:127)
            constexpr float kDecay[12] = { 2.078795764e-01f, 4.321391826e-02f, 8.983291021e-03f, 1.867442732e-03f, 3.882032039e-04f,
                                           8.069951757e-05f, 1.677578152e-05f, 3.487342356e-06f, 7.249472516e-07f, 1.507017275e-07f,
                                           3.132781128e-08f, 6.512412136e-09f };
            // Both windowed sequences go to the exchange buffer in natural (skewed) order as the packed input of FFT-alpha,
            // z[n] = x[n] w[n] + i y[n] w[n]: the transform's strided gather is then one 8-byte load per point.
            if (kPackFilter)
            {
                // (two samples per instruction: the neighbour's decaying contribution, the ramp, and each sample's two sequences by its ramp value)
                #pragma unroll
                for (int j = 0; j < 16; j += 2)
                {
                    float2 y2 = make_float2 (ys[j], ys[j + 1]);
                    if (j < 12) y2 = f2fma (make_float2 (kDecay[j], kDecay[j + 1]), make_float2 (yin, yin), y2);
                    // Bartlett ramp at n = n0 + j (RealTimeAudioAnalysis.h:148-149: w[n] = n * 2/N, w[N/2 + n] = 1 - n * 2/N): all 16
                    // samples lie in the same half and every ramp value is a multiple of 2/N in [0, 1], exact in fp32
                    // (what is stored is z / 2 -- see the split below)
                    const float2 w2 = f2fma (make_float2 ((float) j, (float) (j + 1)), make_float2 (wseg_d, wseg_d), make_float2 (wseg_0, wseg_0));
                    float2* zp = &sm.ex[(t >> 4) * D::ROW + 17 * (t & 15) + j];                                                   // tpos (16 t + j)
                    zp[0] = f2mul (make_float2 (xg[j], y2.x), make_float2 (w2.x, w2.x));
                    zp[1] = f2mul (make_float2 (xg[j + 1], y2.y), make_float2 (w2.y, w2.y));
                }
            }
            else
            {
                #pragma unroll
                for (int j = 0; j < 16; ++j)
                {
                    if (j < 12) ys[j] = fmaf (kDecay[j], yin, ys[j]);
                    // Bartlett ramp at n = n0 + j (RealTimeAudioAnalysis.h:148-149: w[n] = n * 2/N, w[N/2 + n] = 1 - n * 2/N): all 16
                    // samples lie in the same half and every ramp value is a multiple of 2/N in [0, 1], exact in fp32
                    // (packed multiply: both sequences by the same ramp value.  What is stored is z / 2 -- see the split below)
                    const float w = fmaf ((float) j, wseg_d, wseg_0);
                    sm.ex[(t >> 4) * D::ROW + 17 * (t & 15) + j] = f2mul (make_float2 (__fmul_rn (xs[j], gain), ys[j]), make_float2 (w, w));   // tpos (16 t + j)
                }
            }
        }
        __syncthreads();

        // =========================== FFT-alpha: z = x w + i onepole (x) w ==============================
        // Both windowed sequences are real: one complex transform carries B = FFT (x w) (spectral features) and
        // C = FFT (filtered x w) (pitch), separated afterwards by conjugate symmetry.
        V16 io;
        #pragma unroll
        for (int q = 0; q < Q1; ++q)
            #pragma unroll
            for (int n1 = 0; n1 < R1; ++n1)
                io.v[q * R1 + n1] = sm.ex[n1 * D::ROW + phys (T * q + t)];                  // tpos (n1 * 256 + m)
        // no barrier: stage 1 is in place per thread (it stores to ex[k1 * ROW + phys (m)], exactly the slots
        // ex[n1 * ROW + phys (m)] this thread has just read)
        if (kEvenBeta) fft_core_pruned<R1> (io, t, false);
        else           fft_core<R1> (io, t);
        __syncthreads();                                            // Z[k] = B[k] + i C[k] is complete, at zpos (k)

        // previous non-silent spectrum of this thread's bins: issued now, consumed in pass 1 (L2 latency hidden by the split)
        float4 p0 = make_float4 (0.0f, 0.0f, 0.0f, 0.0f), p1 = p0;
        if (have_prev)
        {
            p0 = *reinterpret_cast<const float4*> (&prev_g[b0]);
            p1 = *reinterpret_cast<const float4*> (&prev_g[b0 + 4]);
        }
        // Split for this thread's own 8 consecutive bins k: Z[k] = B[k] + i C[k], conj Z[N-k] = B[k] - i C[k]
        //   Re B = (Zk.x + Zn.x) / 2   Im B = (Zk.y - Zn.y) / 2   Re C = (Zk.y + Zn.y) / 2     (the buffer holds Z / 2)
        // Re B stays in registers for the spectral passes; P[k] = Re C[k]^2 (PitchAnalyser.h:97-104, imaginary part
        // cleared) goes to the P / Re A array as the imaginary input of FFT-beta.
        // Power mode (SP): |B| takes Re B's place, Im C = (Re Z[N-k] - Re Z[k]) / 2 and P = |C|^2.
        float cr[8];
        float rawmax = 0.0f;     // SpectralCharacteristics.h:153: max |buf[j]|, j < M, over the interleaved Re/Im floats = bins k < M/2
        float psum = 0.0f;       // sum of P^2 over the lower half: sets the power-of-two scale P is transformed at
        {
            float pq[8];
            #pragma unroll
            for (int j = 0; j < 8; ++j)
            {
                const float2 zk = sm.ex[zb_own + zrun<R1> (j)];                                // Z[k], k = b0 + j
                const float2 zn = sm.ex[j == 0 ? zb_self : zb_mirror + zrun<R1> (8 - j)];      // Z[(N - k) & (N - 1)]
                const float reB = zk.x + zn.x, reC = zk.y + zn.y;
                const float imB = zk.y - zn.y;
                if (SP)
                {
                    const float imC = zn.x - zk.x;
                    cr[j] = __fsqrt_rn (fmaf (reB, reB, __fmul_rn (imB, imB)));
                    if (b0 < M / 2) rawmax = fmaxf (rawmax, cr[j]);                              // the odd (Im) slots hold 0
                    pq[j] = fmaf (reC, reC, __fmul_rn (imC, imC));
                }
                else
                {
                    cr[j] = reB;
                    if (b0 < M / 2) rawmax = fmaxf (rawmax, fmaxf (fabsf (reB), fabsf (imB)));
                    pq[j] = __fmul_rn (reC, reC);
                }
                psum = fmaf (pq[j], pq[j], psum);
            }
            *reinterpret_cast<float4*> (&sm.pa[pb0])     = make_float4 (pq[0], pq[1], pq[2], pq[3]);
            *reinterpret_cast<float4*> (&sm.pa[pb0 + 4]) = make_float4 (pq[4], pq[5], pq[6], pq[7]);
            if (t == 0) { const float cm = 2.0f * sm.ex[zpos<R1> (M)].y; sm.pa[sk32 (M)] = __fmul_rn (cm, cm); }      // C[N/2] is real and pairs with itself
            if constexpr (SO)
            {
                // mag[b0 + j] rounded once to fp32 (pass 1 squares the same cr[j] exactly in fp64), every frame, silent or not.
                // Two 16-byte stores per thread, 1 KB contiguous per warp; evict-first (st.global.cs), so that the rows
                // streaming out do not push the stage-1 twiddle table (read through L1 / L2 every frame) out of the caches.
                float4* row = reinterpret_cast<float4*> (p.spec + (size_t) (track * p.n_frames + f) * M + b0);
                __stcs (row,     make_float4 (__fmul_rn (cr[0], cr[0]), __fmul_rn (cr[1], cr[1]), __fmul_rn (cr[2], cr[2]), __fmul_rn (cr[3], cr[3])));
                __stcs (row + 1, make_float4 (__fmul_rn (cr[4], cr[4]), __fmul_rn (cr[5], cr[5]), __fmul_rn (cr[6], cr[6]), __fmul_rn (cr[7], cr[7])));
            }
        }

        // RMS (RealTimeAnalyser.h:207-208)
        double rms_sum = 0.0;
        #pragma unroll
        for (int w = 0; w < NW; w += 2)
        {
            const double2 r2 = *reinterpret_cast<const double2*> (&sm.rms[w]);
            rms_sum += r2.x; rms_sum += r2.y;
        }
        // K1b recomputes both in double for the RMS feature; here they only set the flatness gate, whose margin is reported
        const float rms = __fsqrt_rn ((float) (rms_sum * (1.0 / (double) N)));
        const float log_rms = log10f (__fadd_rn (__fmul_rn (rms, 9.0f), 1.0f));
        const double eps = 0.01 * (double) log_rms;                                               // SpectralCharacteristics.h:108

        // =========================== spectral features, pass 1 ========================================
        ME lprod = me_one();
        {
            const float pr[8] = { p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w };
            double mag_sum = 0.0, weighted = 0.0, flux = 0.0, lhr = 0.0, flat_sum = 0.0;
            double s2 = 0.0, s4 = 0.0;
            const double x0 = ((double) b0 + 0.5) * inv_m;                                        // (bin + 1/2) / M, exact
            int count = 0;
            float maxre = 0.0f;
            // gate margin: the smallest distance of |Re| from sqrt (eps), relative to sqrt (eps) -- a lower bound of the
            // relative gap between Re^2 and eps ((1 + d)^2 - 1 >= d and 1 - (1 - d)^2 >= d), two instructions per bin
            const float eps_f = (float) eps;
            const float gate_s = MG ? __fsqrt_rn (eps_f) : 0.0f;
            const float gate_inv = gate_s > 0.0f ? __fdividef (1.0f, gate_s) : 3.0e38f;
            float gate_d = 3.0e38f;
            double mprod = 1.0; int esum = 0;
            #pragma unroll
            for (int j = 0; j < 8; ++j)
            {
                const int bin = b0 + j;
                const double re = (double) cr[j];
                const double mg = re * re;                                                       // :72-73  Re^2
                const double pm = (double) pr[j] * (double) pr[j];
                const double diff = mg - pm;                                                     // :76-79
                if (kFluxF32Cmp)
                {
                    if (fabsf (cr[j]) > fabsf (pr[j])) flux += diff;                                 // mg > pm: both are exact squares
                }
                else
                {
                    if (diff > 0.0) flux += diff;
                }
                mag_sum += mg;
                if (! kLhrRange && bin <= lower_portion) lhr += mg;                              // :86-87
                if (mg > eps)                                                                    // :89-94
                {
                    flat_sum += mg;
                    count += 1;
                    const ME q = me_from (mg);
                    mprod *= q.m;                                                                // >= 2^-8: no renormalisation needed
                    esum += q.e;
                }
                if (MG) gate_d = fminf (gate_d, fabsf (fabsf (cr[j]) - gate_s));
                const double x = x0 + (double) j * inv_m;                                        // fc / nyquist (:70, :137)
                const double xm = x * mg;
                weighted += xm;
                s2 = fma (x, xm, s2);
                s4 = fma (mg, mg, s4);
                maxre = fmaxf (maxre, fabsf (cr[j]));
            }
            if (kLhrRange)
            {
                if (b0 + 7 <= lower_portion) lhr = mag_sum;                                       // :86-87 (the same additions in the same order)
                else if (b0 <= lower_portion)
                {
                    #pragma unroll
                    for (int j = 0; j < 8; ++j) if (b0 + j <= lower_portion) lhr += (double) cr[j] * (double) cr[j];
                }
            }
            lprod = me_from (mprod); lprod.e += esum;
            // The raw moments cross the lanes in fp64: K1b's spread is S2 - 2 c W1 + c^2 S0, and on a narrowband frame that difference
            // is ~1e-6 of its terms, so fp32 partials of S0, W1, S2 (relative rounding ~6e-8) would leave errors of the order of the
            // spread itself.  S4 takes the fourth fp64 slot, which costs no extra exchange.  The sums of positive terms that feed
            // nothing but a ratio stay fp32; the norm of P rides in their free fourth slot (profiles/r02_v31_ab_psum_always_4096.txt).
            double sd[4] = { mag_sum, weighted, s2, s4 };
            float sf[4] = { (float) flux, (float) lhr, (float) flat_sum, psum };
            warp_sum_t<4> (sd, lane);
            warp_sum_t<4> (sf, lane);
            const int wcount = warp_addi (count);
            const float wmax = warp_max_nonneg (maxre);
            const float wraw = warp_max_nonneg (rawmax);
            const float wps = __shfl_sync (0xffffffffu, sf[0], 3);                                  // slot 3's total lives in lanes = 3 mod 4
            float wmar = 1.0f;
            if (MG) wmar = warp_min_nonneg (fminf (gate_d * gate_inv, 0.5f));
            // inclusive warp scan of the extended-range product, in bin order; the mantissa in fp32 (the exponent is an integer,
            // and the product only feeds pow (., 1 / count))
            struct { float m; int e; } incf = { (float) lprod.m, lprod.e };                      // m in [0.5, 1]
            #pragma unroll
            for (int off = 1; off < 32; off <<= 1)
            {
                const float om = __shfl_up_sync (0xffffffffu, incf.m, off); const int oe = __shfl_up_sync (0xffffffffu, incf.e, off);
                if (lane >= off)
                {
                    float m = om * incf.m; int e = oe + incf.e;                                   // m in [0.25, 1]
                    if (m < 0.5f) { m *= 2.0f; e -= 1; }
                    incf.m = m; incf.e = e;
                }
            }
            ME inc; inc.m = (double) incf.m; inc.e = incf.e;
            ME exc; exc.m = __shfl_up_sync (0xffffffffu, inc.m, 1); exc.e = __shfl_up_sync (0xffffffffu, inc.e, 1);
            if (lane == 0) exc = me_one();
            lprod = exc;                                                                         // lane-exclusive prefix within the warp
            // The warp's partials leave for K1b from here (the frame record's WarpPart of this warp, one 80-byte run); only what this CTA's own
            // threads need -- the magnitude sum, the largest |Re|, the norm of P and the product's warp totals -- also goes
            // through shared memory.  After the transposed butterflies lane l holds the warp totals of slot warp_sum_slot<4> (l) of both
            // arrays: sd 0 S0, 1 W1, 2 S2, 3 S4; sf 0 flux, 1 lhr, 2 flat_sum, 3 the norm of P (not recorded).
            WarpPart* wp = &rec_w[warp];
            if (lane == 31)
            {
                *reinterpret_cast<double2*> (&sm.scan[warp]) = make_double2 (inc.m, __hiloint2double (__float_as_int ((float) inc.m), inc.e));
                wp->scan_m = inc.m; wp->scan_e = inc.e;
            }
            if (lane < 4) wp->p1d[warp_sum_slot<4> (lane)] = sd[0];
            else if (lane < 7) wp->p1f[warp_sum_slot<4> (lane)] = sf[0];
            if (lane == 0)
            {
                wp->count = wcount; wp->rawmax = wraw;
                // S0: every thread needs the magnitude sum
                *reinterpret_cast<double2*> (&sm.p1s[warp]) = make_double2 (sd[0], __hiloint2double (__float_as_int (wps), __float_as_int (wmax)));
                if (MG) sm.fmins[0][warp] = wmar;
            }
        }
        __syncthreads();
        double mag_sum_acc = 0.0;
        float maxre_all = 0.0f, psum_all = 0.0f;
        ME prefix = me_one();
        float pfm = 0.5f; int pfe = 1;
        // every thread needs the magnitude sum (silence gate), the largest |Re| (exponent budget below) and the norm of P;
        // everything else of the pass has already left for K1b as per-warp partials
        #pragma unroll
        for (int w = 0; w < NW; ++w)
        {
            const double2 sl = *reinterpret_cast<const double2*> (&sm.p1s[w]);                    // one LDS.128: { s0, (maxre, psum) }
            mag_sum_acc += sl.x;
            maxre_all = fmaxf (maxre_all, __int_as_float (__double2loint (sl.y)));
            psum_all += __int_as_float (__double2hiint (sl.y));
        }
        const double mag_sum = (double) mag_sum_acc;
        #pragma unroll 1
        for (int w = 0; w < warp; ++w)
        {
            const double2 sl = *reinterpret_cast<const double2*> (&sm.scan[w]);
            const float wm = __int_as_float (__double2hiint (sl.y));                              // the warp total's fp32 mantissa rides in the slot's spare word
            pfm *= wm; pfe += __double2loint (sl.y);
            if (pfm < 0.5f) { pfm *= 2.0f; pfe -= 1; }
        }
        prefix.m = (double) pfm; prefix.e = pfe;
        prefix = me_mul (prefix, lprod);
        const double maxmag = (double) maxre_all * (double) maxre_all;
        const bool silent = ! (mag_sum > 0.05);                                                   // :121-123
        // how far 8 gated bins can move the exponent of the running flatness product: every gated magnitude lies in
        // (eps, maxmag], so its exponent is bounded by the larger of the two ends' (CTA-uniform, no per-bin bookkeeping)
        int e_budget = 0;
        if (maxmag > 0.0)
        {
            const int e_hi = ((__double2hiint (maxmag) >> 20) & 0x7ff) - 1022;
            const int e_lo = eps > 0.0 ? ((__double2hiint (eps) >> 20) & 0x7ff) - 1022 : -310;   // squares of fp32 values are >= 2^-298
            e_budget = 8 * (max (abs (e_hi), abs (e_lo)) + 2);
        }

        // =========================== flatness range events ==============================================
        {
            // The running product can leave the normal fp64 range inside this thread's bins only if its prefix is still in
            // range and the exponent budget of its bins reaches a limit.  Such a thread runs the reference's own sequential IEEE
            // multiply (:92) over its 8 bins, from registers, starting at its prefix (which equals the reference's running
            // product up to rounding as long as no earlier thread saw an event).  If the product really left the normal range
            // (entered the denormal band, reached 0 or inf) the thread offers its product; the record stage takes the offer
            // of the earliest such thread and keeps multiplying through the rest of the spectrum -- gradual underflow, sticky
            // 0 / inf and a recovery from the denormal band come out exactly as in the reference.
            unsigned ev_code = 0xffffffffu;
            double ev_prod = 0.0;
            if (prefix.e < 1025 && prefix.e > -1022 && (prefix.e + e_budget >= 1025 || prefix.e - e_budget <= -1022))
            {
                double prod = ldexp_normal (prefix.m, prefix.e);
                bool left = false;
                #pragma unroll
                for (int j = 0; j < 8; ++j)
                {
                    const double mg = (double) cr[j] * (double) cr[j];
                    if (mg > eps)
                    {
                        prod *= mg;
                        const int ef = (__double2hiint (prod) >> 20) & 0x7ff;             // 0: zero / denormal, 0x7ff: inf
                        left = left || ef == 0 || ef == 0x7ff;
                    }
                }
                if (left) { ev_code = (unsigned) t; ev_prod = prod; }
            }
            const unsigned wev = warp_minu (ev_code);
            if (lane == 0) sm.ucodes[warp] = wev;
            if (ev_code != 0xffffffffu && ev_code == wev) sm.ev_prod[warp] = ev_prod;             // the warp's earliest event thread
        }
        if (t == 0)
        {
            // the part of the spectral record every thread already holds (the reductions follow after the next transform)
            rec->rms_sum = rms_sum; rec->mag_sum = mag_sum; rec->maxmag = maxmag; rec->have_prev = have_prev ? 1.0f : 0.0f;
        }
        if (! silent)
        {
            if (! have_prev)
            {
                float* fs = p.first_spec + (track * p.n_chunks + chunk) * (long) M;
                *reinterpret_cast<float4*> (&fs[b0])     = make_float4 (cr[0], cr[1], cr[2], cr[3]);
                *reinterpret_cast<float4*> (&fs[b0 + 4]) = make_float4 (cr[4], cr[5], cr[6], cr[7]);
            }
            *reinterpret_cast<float4*> (&prev_g[b0])     = make_float4 (cr[0], cr[1], cr[2], cr[3]);       // :138 prev <- current
            *reinterpret_cast<float4*> (&prev_g[b0 + 4]) = make_float4 (cr[4], cr[5], cr[6], cr[7]);
        }
        if (! silent && ! have_prev) { have_prev = true; first_nonsilent = f; }


        // =========================== FFT-beta: z = x + i 2^k P ==========================================
        // A = FFT (x) feeds the harmonic features through its real part only, and the reference's inverse transform of
        // the real, even sequence P (PitchAnalyser.h:120) is, up to 1/N, the real and even D = FFT (P).  Packed as
        // Z = A + i D:  Re Z = Re A directly, and Im Z[s] + Im Z[N-s] = 2 D[s] because Im A is odd.  P is scaled by a
        // power of two that matches its L2 norm to the frame's (an fp32 FFT's rounding noise is relative to the L2 norm
        // of what it transforms): neither sequence's noise then rises above a small multiple of its own (the lag search is invariant to the scale, cnd = d^2 s / sum).
        // Parity mode: nothing reads Im A, so the transform takes the even part of the frame, e[n] = (x[n] + x[(N - n) & (N - 1)]) / 2,
        // in place of x: Re Z = FFT (e) = Re A, Im Z = 2^k D, and Z is even.  Only the rows k1 <= R1 / 2 of the spectrum are
        // computed (fft_core_pruned); bins and lags of the other rows are read at N - k.  The power mode needs Im A and
        // transforms x.
        {
            float pscale = 1.0f;
            if (psum_all > 0.0f && psum_all < 3.0e38f && rms_sum > 0.0)
            {
                const int e_r = ((__double2hiint (rms_sum) >> 20) & 0x7ff) - 1023;                 // ||x||^2   ~ 2^e_r
                const int e_p = (int) ((__float_as_uint (psum_all) >> 23) & 0xff) - 127;          // ||P||^2/2 ~ 2^e_p
                int k2 = (e_r >> 1) - (e_p >> 1) + 1;                                             // ||2^k P|| = (1 .. 8) ||x||
                k2 = max (-120, min (120, k2));
                pscale = __int_as_float ((k2 + 127) << 23);
            }
            // sample a0 + t + c of the ring and P[c + t] (c < M) or P[N - c - t] (P is even: P[N - n] = P[n]); every c is a
            // multiple of 32, so the skewed positions are a per-thread base plus a compile-time offset (ring: modulo the ring)
            const int rg = (int) ((a0 + t) >> 5) & (N / 32 - 1), rl = (int) ((a0 + t) & 31);
            const int pa_up = 36 * warp + lane;                                                   // sk32 (c + t) - 36 (c / 32)
            const int pa_dn = -36 * warp - lane - (lane ? 4 : 0);                                 // sk32 (N - c - t) - 36 ((N - c) / 32)
            // parity mode: the mirror sample a0 + N - c - t of the ring, from the per-thread base a0 - t
            const int rg2 = (int) ((a0 - t) >> 5) & (N / 32 - 1), rl2 = (int) ((a0 - t) & 31);
            const float hg = 0.5f * gain;
            if (kEvenBeta && NB <= 4)
            {
                // as below; the mirrors of quarter g lie in quarter 3 - g of the window, one wrapped base per quarter (ml), except
                // that of c = g N / 4 for thread 0: sample (4 - g) N / 4 of the window, which thread 0 loads as its own sample of
                // quarter (4 - g) mod 4
                float xo[Q1 * R1];
                #pragma unroll
                for (int g = 0; g < 4; ++g)
                {
                    const float* rq = sm.ring + 36 * ((rg + g * (N / 128)) & (N / 32 - 1)) + rl;
                    #pragma unroll
                    for (int q = 0; q < Q1; ++q)
                        #pragma unroll
                        for (int i = 0; i < R1 / 4; ++i)
                            xo[q * R1 + g * (R1 / 4) + i] = rq[36 * ((i * 256 + T * q) / 32)];
                }
                #pragma unroll
                for (int g = 0; g < 4; ++g)
                {
                    const float* ml = sm.ring + 36 * ((rg2 + (4 - g) * (N / 128) - 1) & (N / 32 - 1)) + rl2;    // sample a0 - t + (4 - g) N / 4 - 32
                    #pragma unroll
                    for (int q = 0; q < Q1; ++q)
                        #pragma unroll
                        for (int i = 0; i < R1 / 4; ++i)
                        {
                            const int n1 = g * (R1 / 4) + i;
                            const int c = n1 * 256 + T * q, cq = c - g * (N / 4);
                            const int pidx = (c < M) ? pa_up + 36 * (c / 32) : pa_dn + 36 * ((N - c) / 32);
                            float xm;
                            if (cq != 0)     xm = ml[-36 * ((cq - 32) / 32)];
                            else if (t != 0) xm = ml[36];
                            else             xm = xo[((4 - g) & 3) * (R1 / 4)];
                            io.v[q * R1 + n1] = f2mul (make_float2 (xo[q * R1 + n1] + xm, sm.pa[pidx]), make_float2 (hg, pscale));
                        }
                }
            }
            else if (kEvenBeta)
            {
                #pragma unroll
                for (int q = 0; q < Q1; ++q)
                    #pragma unroll
                    for (int n1 = 0; n1 < R1; ++n1)
                    {
                        const int c = n1 * 256 + T * q;
                        const int pidx = (c < M) ? pa_up + 36 * (c / 32) : pa_dn + 36 * ((N - c) / 32);
                        const int ridx = 36 * ((rg + c / 32) & (N / 32 - 1)) + rl;
                        const int midx = 36 * ((rg2 + (N - c) / 32) & (N / 32 - 1)) + rl2;
                        io.v[q * R1 + n1] = f2mul (make_float2 (sm.ring[ridx] + sm.ring[midx], sm.pa[pidx]), make_float2 (hg, pscale));
                    }
            }
            else if (NB <= 4)
            {
                // the window starts at a multiple of the hop: with hop >= N / 4 the ring wraps at a multiple of N / 4 samples, never
                // inside a quarter of the window -- one wrapped base per quarter, compile-time offsets inside it
                #pragma unroll
                for (int g = 0; g < 4; ++g)
                {
                    const float* rq = sm.ring + 36 * ((rg + g * (N / 128)) & (N / 32 - 1)) + rl;
                    #pragma unroll
                    for (int q = 0; q < Q1; ++q)
                        #pragma unroll
                        for (int i = 0; i < R1 / 4; ++i)
                        {
                            const int n1 = g * (R1 / 4) + i;
                            const int c = n1 * 256 + T * q;
                            const int pidx = (c < M) ? pa_up + 36 * (c / 32) : pa_dn + 36 * ((N - c) / 32);
                            io.v[q * R1 + n1] = f2mul (make_float2 (rq[36 * ((c - g * (N / 4)) / 32)], sm.pa[pidx]), make_float2 (gain, pscale));
                        }
                }
            }
            else
            {
                #pragma unroll
                for (int q = 0; q < Q1; ++q)
                    #pragma unroll
                    for (int n1 = 0; n1 < R1; ++n1)
                    {
                        const int c = n1 * 256 + T * q;
                        const int pidx = (c < M) ? pa_up + 36 * (c / 32) : pa_dn + 36 * ((N - c) / 32);
                        const int ridx = 36 * ((rg + c / 32) & (N / 32 - 1)) + rl;
                        io.v[q * R1 + n1] = f2mul (make_float2 (sm.ring[ridx], sm.pa[pidx]), make_float2 (gain, pscale));
                    }
            }
        }
        // No barrier here: stage 1 of the transform stores to this thread's own slots of the exchange buffer, which nobody
        // reads between the barrier above (the split is complete) and the barrier inside the transform.
        if (kEvenBeta) fft_core_pruned<R1> (io, t, true);
        else           fft_core<R1> (io, t);
        // (the record of this frame is written after the frame's last barrier, one part per warp)
        __syncthreads();
        // The flatness product's continuation (record stage, below) starts from the spectrum bins behind the earliest event
        // thread: its warp fetches the first 32 of them now, from the spectrum stored before the transform.
        float ev_pf = 0.0f;
        if (warp == kRoleFlat)
        {
            const unsigned ev = warp_minu (lane < NW ? sm.ucodes[lane] : 0xffffffffu);
            const int b = 8 * ((int) ev + 1) + lane;
            if (ev != 0xffffffffu && ! silent && b < M) ev_pf = prev_g[b];
        }
        // every read of the ring for this frame is complete (filter pass, gather of FFT-beta): prefetch the next hop; it
        // lands during the pitch / harmonic passes
        if (f + 1 < f_end)
        {
            const long jn = j_new + 1;
            const int base = (int) ((jn * H) & (N - 1));
            const float* g = src + (jn - p.first_hop) * H;
            // (the skewed ring takes the block as 16-byte pieces, one or two per thread: asynchronous copies without register
            // staging -- LDGSTS -- whose completion arrives at the mbarrier the next frame waits on.  A bulk copy per 128-byte run
            // was measured 5 % slower at N = 2048 / 1024: 32 small TMA requests per frame cost more than the conflicts they remove)
            if (p.use_bulk) { _Pragma ("unroll 1") for (int k = 4 * t; k < H; k += 4 * T) cp_async16 (&sm.ring[sk32 (base + k)], g + k); }
            else            { _Pragma ("unroll 1") for (int i = t; i < H; i += T) sm.ring[sk32 (base + i)] = g[i]; }
            cp_async_arrive (&sm.mbar);
        }

        // =========================== pitch: cumulative normalised difference + lag search ==============
        // workf holds d[s] (kept for the margins), workg receives cnd[s]; each thread owns s = 16 t .. 16 t + 15
        float av[16];                                                                             // ac[s] = d^2 s (PitchAnalyser.h:122-123)
        float dv[MG ? 16 : 1];                                                                    // d[s]: only the margins look at it again
        double seg_exc;
        {
            const float s0f = (float) (16 * t);
            float runf = 0.0f;
            // two lags per packed instruction: the same values except the order of a thread's 16-term run sum
            float2 run2 = make_float2 (0.0f, 0.0f);
            #pragma unroll
            for (int j = 0; j < 16; j += 2)
            {
                float2 d2;
                if (! kEvenBeta)
                {
                    // Z[s] + Z[N - s]: 2 * 2^k * D[s], two lags per instruction
                    const float2 za = make_float2 (sm.ex[zl_own + zrun<R1> (j)].y, sm.ex[zl_own + zrun<R1> (j + 1)].y);
                    const float2 zb = make_float2 (sm.ex[j == 0 ? zl_self : zl_mirror + zrun<R1> (16 - j)].y, sm.ex[zl_mirror + zrun<R1> (15 - j)].y);
                    d2 = f2add (za, zb);
                }
                else
                {
                    // Im Z[s] = 2^k D[s] (half the value above: cnd and its margins do not depend on the scale); the row of lag
                    // s = 16 t + j is j mod R1, and a lag in a row that was not computed reads its mirror N - s
                    const int j1 = j + 1;
                    d2 = make_float2 (sm.ex[(j & (R1 - 1)) > R1 / 2 ? zl_mirror + zrun<R1> (16 - j) : zl_own + zrun<R1> (j)].y,
                                      sm.ex[(j1 & (R1 - 1)) > R1 / 2 ? zl_mirror + zrun<R1> (16 - j1) : zl_own + zrun<R1> (j1)].y);
                }
                if (MG) { dv[j] = d2.x; dv[j + 1] = d2.y; }
                const float2 s2 = f2add (make_float2 (s0f, s0f), make_float2 ((float) j, (float) (j + 1)));
                const float2 a2 = f2mul (f2mul (d2, d2), s2);                                     // s = 0 contributes 0
                av[j] = a2.x; av[j + 1] = a2.y;
                run2 = f2add (run2, a2);
            }
            runf = run2.x + run2.y;
            // Re A of this thread's 8 bins moves to the P / Re A array (P was consumed by the transform).  Power mode: |A|, with
            // Im A[k] = (Im Z[k] - Im Z[N-k]) / 2 -- Im A is odd and 2^k D even, so D cancels.
            {
                float ra[8];
                #pragma unroll
                for (int j = 0; j < 8; ++j)
                {
                    if (SP)
                    {
                        const float2 zk = sm.ex[zb_own + zrun<R1> (j)];
                        const float imA = 0.5f * (zk.y - sm.ex[j == 0 ? zb_self : zb_mirror + zrun<R1> (8 - j)].y);
                        ra[j] = __fsqrt_rn (fmaf (zk.x, zk.x, __fmul_rn (imA, imA)));
                    }
                    else if (! kEvenBeta) ra[j] = sm.ex[zb_own + zrun<R1> (j)].x;
                    else
                    {
                        // a bin in a row that was not computed reads its mirror N - k.  The row of bin b0 + j is j mod R1, except
                        // at N = 4096, where the run of an odd thread covers rows 8 .. 15
                        const bool mirror = R1 == 16 ? (j > 0 && (t & 1)) : (j & (R1 - 1)) > R1 / 2;
                        ra[j] = sm.ex[mirror ? zb_mirror + zrun<R1> (8 - j) : zb_own + zrun<R1> (j)].x;
                    }
                }
                *reinterpret_cast<float4*> (&sm.pa[pb0])     = make_float4 (ra[0], ra[1], ra[2], ra[3]);
                *reinterpret_cast<float4*> (&sm.pa[pb0 + 4]) = make_float4 (ra[4], ra[5], ra[6], ra[7]);
            }
            // warp scan of the cumulative sum in fp32 (the reference runs this sum in fp32 sequentially, :138-145)
            float inc = runf;
            #pragma unroll
            for (int off = 1; off < 32; off <<= 1)
            {
                const float o = __shfl_up_sync (0xffffffffu, inc, off);
                if (lane >= off) inc += o;
            }
            const float excf = __shfl_up_sync (0xffffffffu, inc, 1);
            seg_exc = lane == 0 ? 0.0 : (double) excf;
            if (lane == 31) sm.pscan[warp] = inc;
            if (MG && t == 0) sm.d0 = dv[0];
        }
        __syncthreads();
        unsigned first_cross = 0xffffffffu, nd_mask = 0u, wfc, wbest;
        {
            // the segment's running sum starts from the fp32 sum of the preceding warps' fp32 totals
            float sumf = 0.0f;
            #pragma unroll
            for (int w = 0; w < NW; w += 2)
            {
                const float2 p2 = *reinterpret_cast<const float2*> (&sm.pscan[w]);
                if (w < warp) sumf += p2.x;
                if (w + 1 < warp) sumf += p2.y;
            }
            sumf += (float) seg_exc;
            float best = 100.0f;
            unsigned cross = 0u;
            float c_before = 0.0f;
            #pragma unroll
            for (int j = 0; j < 16; ++j)
            {
                sumf += av[j];
                float c = (sumf != 0.0f) ? __fmul_rn (av[j], rcp_approx (sumf)) : 0.0f;          // :146-154
                if (j == 0 && t == 0) c = 1.0f;                                                   // :141
                workg[17 * t + j] = c;
                if (MG) workf[17 * t + j] = dv[j];                                                // every read of Z is behind the barrier above
                if (j > 0 && ! (c < c_before)) nd_mask |= 1u << (j - 1);          // the descent (:178) stops at j - 1
                c_before = c;
                if (j >= 2 || t != 0)                                                             // the search starts at s = 2 (:169)
                {
                    best = fminf (best, c);                                                       // :171-175 (its index only matters when no lag crosses: found then)
                }
            }
            // :176 some lag of this thread is under the threshold iff its minimum is: only then (few threads of a frame) look for the first
            if (best < 0.01f)
            {
                #pragma unroll
                for (int j = 15; j >= 0; --j)
                    if ((j >= 2 || t != 0) && workg[17 * t + j] < 0.01f) cross = 1u << j;        // (this thread's own stores)
            }
            sm.ndm[t] = (unsigned short) nd_mask;
            if (cross != 0u) first_cross = (unsigned) (16 * t + __ffs ((int) cross) - 1);
            // smallest cnd of the warp (cnd >= 0 orders like its bit pattern)
            wfc = warp_minu (first_cross);
            wbest = warp_minu (__float_as_uint (best));
        }
        // harmonic pass A (independent of the pitch): sum and max of Re A ^2 (HarmonicCharacteristics.h:61-69).  The three
        // neighbours the peak test needs from other threads (bins b0 - 2, b0 - 1, b0 + 8) are fetched now: after the next
        // barrier every thread overwrites its own 8 bins of the array with the normalised magnitudes.
        float ar[11];
        {
            const float4 a0v = *reinterpret_cast<const float4*> (&sm.pa[pb0]);
            const float4 a1v = *reinterpret_cast<const float4*> (&sm.pa[pb0 + 4]);
            ar[2] = a0v.x; ar[3] = a0v.y; ar[4] = a0v.z; ar[5] = a0v.w; ar[6] = a1v.x; ar[7] = a1v.y; ar[8] = a1v.z; ar[9] = a1v.w;
            ar[0] = (b0 >= 2) ? sm.pa[sk32 (b0 - 2)] : 0.0f;
            ar[1] = (b0 >= 1) ? sm.pa[sk32 (b0 - 2) + 1] : 0.0f;
            ar[10] = (b0 + 8 < M) ? sm.pa[sk32 (b0 + 8)] : 0.0f;
            float hmaxre = 0.0f;
            float hsf = 0.0f;
            #pragma unroll
            for (int j = 0; j < 8; ++j) { hsf = fmaf (ar[2 + j], ar[2 + j], hsf); hmaxre = fmaxf (hmaxre, fabsf (ar[2 + j])); }
            double s1[1] = { (double) warp_sumf (hsf) };
            const float wm = warp_max_nonneg (hmaxre);
            if (lane == 0) *reinterpret_cast<float4*> (&sm.lags[warp]) = make_float4 ((float) s1[0], wm, __uint_as_float (wfc), __uint_as_float (wbest));
        }
        __syncthreads();
        // ---- every thread now derives the lag on its own (all control flow below is uniform across the CTA) -----------
        unsigned s0 = 0xffffffffu;
        unsigned gbest = 0xffffffffu;                              // bit pattern of the smallest cnd of the search range
        float hmaxre = 0.0f;
        float hsum_acc = 0.0f;
        #pragma unroll
        for (int w = 0; w < NW; ++w)
        {
            const float4 sl = *reinterpret_cast<const float4*> (&sm.lags[w]);                     // one LDS.128: { hsum, largest |Re A|, first_cross, best }
            s0 = min (s0, __float_as_uint (sl.z));
            gbest = min (gbest, __float_as_uint (sl.w));
            hsum_acc += sl.x;
            hmaxre = fmaxf (hmaxre, sl.y);
        }
        const double hsum = (double) hsum_acc;
        const double hmax = (double) hmaxre * (double) hmaxre;
        const bool crossed = (s0 != 0xffffffffu);
        const float e_abs = MG ? 1.0e-6f * fabsf (sm.d0) : 0.0f;
        int lag_i;                                                   // integer lag, -1 when the search found nothing (:165,188)
        float pm = 1.0f;
        if (crossed)
        {
            // end of the descending run that starts at s0 (:178-181): walk the per-segment "not descending" masks
            int seg = (int) (s0 >> 4), j0 = (int) (s0 & 15u);
            int s_end;
            #pragma unroll 1
            for (;;)
            {
                const unsigned m = ((unsigned) sm.ndm[seg]) >> j0;                      // positions j0 .. 14 of this segment
                if (m != 0u) { s_end = 16 * seg + j0 + __ffs ((int) m) - 1; break; }
                const int s = 16 * seg + 15;                                          // position 15 looks into the next segment
                if (s + 1 >= N || ! (workg[phys (s + 1)] < workg[phys (s)])) { s_end = s; break; }
                ++seg; j0 = 0;
            }
            // getInterpolatedValleyFromCumulativeDifferenceLagEstimate (:192-203): the parabolic branch is unreachable
            const int right = s_end + 1;
            const float c_end = workg[phys (s_end)];
            const float c_right = (right < N) ? workg[phys (right)] : 0.0f;          // cnd[N] = Im part of lag 0 = 0
            lag_i = (c_end <= c_right) ? s_end : right;
            // margins (diagnostics), spread over the whole CTA: the threshold tests s = 2 .. s0 (:176) ...
            // (work is dealt from the last warp backwards: the low lags meet the warp that has no peaks to process below)
            if (MG)
            {
                const int tr = (t + 32) & (T - 1);
                #pragma unroll 1
                for (int s = 2 + tr; s <= (int) s0; s += T)
                {
                    const float c = workg[phys (s)];
                    pm = fminf (pm, noisy_margin (c, cnd_uncertainty (c, workf[phys (s)], e_abs), 0.01f, 0.0f));
                }
                // ... and every comparison the descent made, (s - 1, s) for s = s0 + 1 .. s_end + 1
                const int s_hi = min (s_end + 1, N - 1);
                #pragma unroll 1
                for (int s = (int) s0 + 1 + tr; s <= s_hi; s += T)
                {
                    const float c = workg[phys (s)], cp = workg[phys (s - 1)];
                    const float u = cnd_uncertainty (c, workf[phys (s)], e_abs);
                    const float up = cnd_uncertainty (cp, workf[phys (s - 1)], e_abs);
                    pm = fminf (pm, noisy_margin (c, u, cp, up));
                }
            }
        }
        else
        {
            // No lag crossed the threshold (:188-189, rare): the lag is the first strict global minimum (:171-175), the smallest
            // index among the lags that hold the smallest value.  One more block reduction, in this CTA-uniform branch only.
            unsigned mine = 0xffffffffu;
            #pragma unroll
            for (int j = 15; j >= 0; --j)
                if ((j >= 2 || t != 0) && __float_as_uint (workg[17 * t + j]) == gbest) mine = (unsigned) (16 * t + j);
            const unsigned wmine = warp_minu (mine);
            if (lane == 0) sm.ugidx[warp] = wmine;
            __syncthreads();
            unsigned gidx = 0xffffffffu;
            #pragma unroll
            for (int w = 0; w < NW; ++w) gidx = min (gidx, sm.ugidx[w]);
            lag_i = (gidx == 0xffffffffu) ? -1 : (int) gidx;
            // no crossing: every threshold test was false; runner-up of the global minimum for its margin
            if (MG)
            {
                float second = 100.0f;
                #pragma unroll 2
                for (int j = (t == 0 ? 2 : 0); j < 16; ++j)
                {
                    const float c = workg[17 * t + j];
                    pm = fminf (pm, noisy_margin (c, cnd_uncertainty (c, workf[17 * t + j], e_abs), 0.01f, 0.0f));
                    if (16 * t + j != (int) gidx) second = fminf (second, c);
                }
                const float wsec = warp_min_nonneg (second);
                if (lane == 0) sm.pmins[1][warp] = wsec;
            }
        }
        if (MG)
        {
            const float wpm = warp_min_nonneg (pm);
            if (lane == 0) sm.pmins[0][warp] = wpm;
        }
        // The frame's last block barrier: every read of the cnd values (the exchange buffer, which the next frame's filter pass
        // overwrites) and of the descent masks (whose storage the record stage reuses) is behind it.  The peak loop below -- a
        // thread-dependent number of peaks -- and the record stage then run into the next frame's filter pass without another
        // barrier: their imbalance is absorbed once, at the barrier behind that pass, not twice.  What they read (this thread's
        // registers, the P / Re A array, per-warp slots of earlier phases) is not written again before the next frame's pass 1.
        __syncthreads();
        // The harmonic and sub-octave bins of f0 = sample rate / lag come from a table built on the host with the reference's
        // own double arithmetic (PitchAnalyser.h:57, HarmonicCharacteristics.h:158-185): slot 0 stands for lag -1
        const int lag_slot = lag_i < 0 ? 0 : lag_i;
        const short* htab = p.her_tab + (size_t) lag_slot * FX_HER_TAB_STRIDE;
        // bin of f0 (:246-249): floor (f0 / frpb) is floor (N / lag) unless the quotient is an exact integer (lag a power of
        // two), where the reference's fp64 rounding decides -- those few values come with the parameters.  No global load
        // sits between the lag and the peak loop.
        int f0_bin = -1;
        if (lag_i > 0) f0_bin = (lag_i & (lag_i - 1)) ? idiv_n<N> (lag_i, rcp_approx ((float) lag_i)) : (int) p.f0bin_pow2[__ffs (lag_i) - 1];
        const int ex_base = __ldg (p.ex_off + lag_slot);          // this lag's entries of the exact-ratio table (used below, rarely)
        int her_bin = -1;
        if (warp == kRoleHer && lane < 18) her_bin = (int) __ldg (&htab[lane]);       // consumed after the next barrier

        // =========================== harmonic features (HarmonicCharacteristics.h:46-106) =============
        const bool hsilent = hsum < 0.005;                                                        // :88
        const double mean_mag = hsum * inv_m;                                                     // :86
        {
            double inharm = 0.0;                // sum of f0Proportion * binMagnitude; the record stage divides by the magnitude sum (:237)
            unsigned pgap = 0xffffffffu, peak_mask = 0u;
            const float mean_f = (float) mean_mag;
            // neighbours bin-2, bin-1, bin+1 (:136-143, loop end exclusive).  The magnitudes are exact squares of fp32 values in
            // fp64, so "a neighbour's magnitude is larger" is decided by |Re| alone; only the test against the mean needs the square.
            float aa[11];
            #pragma unroll
            for (int j = 0; j < 11; ++j) aa[j] = fabsf (ar[j]);
            #pragma unroll
            for (int j = 0; j < 8; ++j)
            {
                const int bin = b0 + j;
                const double mg = (double) ar[2 + j] * (double) ar[2 + j];
                const float mgf = (float) mg;
                if (MG) pgap = min (pgap, ulp_gap (mgf, mean_f));
                if (mg > mean_mag)
                {
                    // edge clamps (:136-137): the neighbour window is [max (bin-2, 0), min (bin+2, M-1))
                    const int lo = bin - 2 > 0 ? bin - 2 : 0;
                    const int hi = bin + 2 < M - 1 ? bin + 2 : M - 1;                             // exclusive
                    const float a = aa[2 + j];
                    bool peak = true;
                    if (bin - 2 >= lo && bin - 2 < hi) { if (MG) pgap = min (pgap, ulp_gap (__fmul_rn (aa[j], aa[j]), mgf)); if (aa[j] > a) peak = false; }
                    if (peak && bin - 1 >= lo && bin - 1 < hi) { if (MG) pgap = min (pgap, ulp_gap (__fmul_rn (aa[j + 1], aa[j + 1]), mgf)); if (aa[j + 1] > a) peak = false; }
                    if (peak && bin + 1 < hi) { if (MG) pgap = min (pgap, ulp_gap (__fmul_rn (aa[j + 3], aa[j + 3]), mgf)); if (aa[j + 3] > a) peak = false; }
                    if (peak) peak_mask |= 1u << j;
                }
            }
            const int npeaks = __popc (peak_mask);
            // calculateInharmonicity (:212-244) over this thread's peaks
            // one peak's term of the inharmonicity sum
            auto peak_term = [&] (int bin) -> double
            {
                if (bin == f0_bin) return 0.0;                                                    // :220
                // bin 0 (:224 start = frpb / 2): the start edge's ratio is exactly twice the end edge's, and that one is N / lag >= 1,
                // so their floors always differ (:232) and the bin contributes nothing
                if (bin == 0) return 0.0;
                const double re = (double) sm.pa[sk32 (bin)];                                     // still Re A
                const double mg = re * re;
                // :223-239 compares floor (higher / lower) for the two edges of the bin, start = bin frpb and end = (bin + 1) frpb,
                // against f0 = sample rate / lag.  Up to an ulp of fp64 rounding these ratios are the rationals bin lag / N
                // (bin above f0's) or N / (bin lag) (below): unless one of them is an exact integer -- where the reference's own
                // rounding decides -- their floors are the integer quotients and the fraction is a remainder, no fp64 division.
                const int pl = bin * lag_i, pl2 = pl + lag_i;
                bool exact_path = false;
                int fa = 0, fb = 1;
                double frac = 0.0;
                if (bin > f0_bin)
                {
                    exact_path = ((pl & (N - 1)) == 0) || ((pl2 & (N - 1)) == 0);
                    fa = pl >> LOG_N; fb = pl2 >> LOG_N;
                    frac = (double) (pl & (N - 1)) * (1.0 / (double) N);                          // the smaller ratio is the start edge's
                }
                else
                {
                    // (not a rare case: a frame analysed at a short lag has every peak below f0's bin)
                    const float plf2 = (float) pl2, r1 = rcp_approx ((float) pl), r2 = rcp_approx (plf2);
                    fa = idiv_n<N> (pl, r1); fb = idiv_n<N> (pl2, r2);
                    const int rem2 = N - fb * pl2;
                    exact_path = (N - fa * pl == 0) || (rem2 == 0);
                    // the smaller ratio is the end edge's: fraction rem2 / pl2 < 1 from the fp32 reciprocal with one residual
                    // correction (relative error ~1e-7 on a term whose sum is compared at 1e-4)
                    const float q0 = (float) rem2 * r2;
                    frac = (double) fmaf (fmaf (-q0, plf2, (float) rem2), r2, q0);
                }
                if (exact_path)
                {
                    // an edge ratio may be an exact integer: the reference's fp64 rounding decides, and its value for this
                    // (lag, bin) comes from the table the host evaluated in the reference's arithmetic
                    const int sh = LOG_N - (__ffs (lag_i) - 1);                                   // log2 (N / gcd (lag, N))
                    int idx;
                    if (bin > f0_bin) idx = (bin & ((1 << sh) - 1)) == 0 ? 2 * (bin >> sh) : 2 * ((bin + 1) >> sh) + 1;
                    else              idx = (bin & (bin - 1)) == 0 ? 2 * (__ffs (bin) - 1) - 26 : 2 * (__ffs (bin + 1) - 1) + 1 - 26;
                    return __ldg (p.ex_tab + (ex_base + idx)) * mg;
                }
                return fa == fb ? frac * mg : 0.0;
            };
            // calculateInharmonicity (:212-244)
            if (lag_i > 0)                                                                        // :98 f0 > 0
            {
                #pragma unroll 1
                while (peak_mask)
                {
                    const int j = __ffs ((int) peak_mask) - 1;
                    peak_mask &= peak_mask - 1u;
                    inharm += peak_term (b0 + j);
                }
            }
            const float pkm = ulps_to_margin (pgap);
            // (the normalised magnitudes of :71-77 are not materialised: their sum is magnitudeSum / maxMagnitude up to fp64
            // rounding, and the few the harmonic energy terms look at are formed from Re A by the record stage)
            double s1[1] = { (double) warp_sumf ((float) inharm) };
            const int wnp = warp_addi (npeaks);
            if (lane == 0) { rec_w[warp].inharm = s1[0]; rec_w[warp].npeaks = wnp; }           // K1b sums the warps' parts
            if (MG) { const float wpk = warp_min_nonneg (pkm); if (lane == 0) sm.fmins[1][warp] = wpk; }
        }
        if (MG) __syncthreads();                     // (the margins' per-warp minima reach the warp that records them)
        // ---- what is left of the frame's record ----------------------------------------------------------------------
        // The sums only K1b looks at left as per-warp partials where they were formed (the record's WarpParts); what remains here are the
        // values every thread holds (lag, harmonic sum and maximum), the 18 harmonic-energy maxima, the margins (MG) and the
        // flatness product's range event, each on its own warp.  No barrier closes the frame: what these parts read (the
        // P / Re A array, per-warp slots of earlier phases) is not written again before the next frame's pass 1.
        {
            const bool ld = lane < NW;
            if (warp == kRoleHer)
            {
                // calculateHarmonicEnergyCharacteristics (:147-198), numLower = 15, numHarmonics = 3 (:94): lane l < 15 is the
                // sub-octave f0 / 2^(l+1), lanes 15..17 are the harmonics 1..3 (bins from the table, -1 = not used: a sub-octave in
                // f0's own bin is skipped (:163-164), harmonics stop at the first bin >= M (:174-175)); the sums are warp reductions
                float mx = -1.0f;                                                                 // "term not used"
                if (her_bin >= 0 && ! hsilent)
                {
                    const int st = her_bin - 2 >= 0 ? her_bin - 2 : 0;
                    const int en = her_bin + 2 < M ? her_bin + 2 : M;
                    // :200-210 maximum of the normalised magnitudes (float) (mag / max) around the bin: the rounding to float is
                    // monotone, so it is the normalised value of the largest |Re A|, which is what the record keeps; K1b
                    // normalises and sums the 18 terms in the reference's order.
                    // (the window [st, en) holds at most bins c - 2 .. c + 1: four independent loads, indices clamped into the window)
                    const float m0 = fabsf (sm.pa[sk32 (her_bin)]), m1 = fabsf (sm.pa[sk32 (max (her_bin - 2, st))]), m2 = fabsf (sm.pa[sk32 (max (her_bin - 1, st))]);
                    const float m3 = fabsf (sm.pa[sk32 (min (her_bin + 1, en - 1))]);
                    mx = fmaxf (fmaxf (m0, m1), fmaxf (m2, m3));
                }
                if (lane < 18) rec->her_mx[lane] = mx;
            }
            if (warp == kRoleHead)
            {
                float pkm = 1.0f, pmm = 1.0f;
                if (MG)
                {
                    pkm = warp_min_nonneg (ld ? sm.fmins[1][lane] : 1.0f);
                    pmm = warp_min_nonneg (ld ? sm.pmins[0][lane] : 1.0f);
                    const float second = warp_min_nonneg (ld ? sm.pmins[1][lane] : 100.0f);
                    if (! crossed) pmm = fminf (pmm, relmargin_f (__uint_as_float (gbest), second));
                }
                if (lane == 0)
                {
                    rec->lag = (float) lag_i; rec->pitch_margin = pmm; rec->peak_margin = pkm;
                    rec->hsum = hsum; rec->hmax = hmax;                                           // K1b divides (:77, :237)
                }
            }
            if (MG && warp == 3 % NW)
            {
                const float flat_margin = warp_min_nonneg (ld ? sm.fmins[0][lane] : 1.0f);
                if (lane == 0) rec->flat_margin = flat_margin;
            }
            if (warp == kRoleFlat)
            {
                // flatness product: without a range event K1b multiplies the warps' totals (flat_state -1); else the offer of the
                // earliest event thread is continued here
                const unsigned evc = ld ? sm.ucodes[lane] : 0xffffffffu;
                const unsigned ev = warp_minu (evc);
                double product = 0.0; float flat_state = -1.0f;
                if (ev != 0xffffffffu)
                {
                    const int ev_warp = __ffs ((int) __ballot_sync (0xffffffffu, evc == ev)) - 1;
                    product = sm.ev_prod[ev_warp];
                    // The reference keeps multiplying (:92).  The spectrum of a non-silent frame is in prev_g (written before the
                    // last transform's barriers); a silent frame reports no flatness at all (:121-123).  32 bins per step: each
                    // lane holds one (a gated-out bin multiplies by exactly 1; the first 32 were fetched right after the
                    // transform), then every lane replays them in order -- the same sequential IEEE products as the reference's.
                    if (! silent)
                    {
                        int b = 8 * ((int) ev + 1);
                        float re_f = ev_pf;
                        #pragma unroll 1
                        for (;;)
                        {
                            double mgl = 1.0;
                            if (b + lane < M) { const double mg = (double) re_f * (double) re_f; if (mg > eps) mgl = mg; }
                            // zero and inf are sticky under multiplication by finite positive magnitudes: test per group of 8
                            sm.ev_chunk[lane] = mgl;
                            __syncwarp();
                            #pragma unroll 1
                            for (int g = 0; g < 32 && product != 0.0 && ! isinf (product); g += 8)
                            {
                                #pragma unroll
                                for (int i = 0; i < 8; ++i) product *= sm.ev_chunk[g + i];
                            }
                            __syncwarp();
                            b += 32;
                            if (b >= M || product == 0.0 || isinf (product)) break;
                            re_f = (b + lane < M) ? prev_g[b + lane] : 0.0f;
                        }
                    }
                    flat_state = (product == 0.0) ? 1.0f : (isinf (product) ? 2.0f : 0.0f);
                }
                if (lane == 0) { rec->product = product; rec->flat_state = silent ? 3.0f : flat_state; if (! MG) rec->flat_margin = 1.0f; }
            }
        }
    }
    __syncthreads();                                                // the last frame's record and ring reads are complete

    // ---- chunk epilogue ----------------------------------------------------------------------------------
    if (t == 0) p.first_idx[track * p.n_chunks + chunk] = first_nonsilent;
    if (f_end == p.n_frames && p.tail_out != nullptr)
    {
        // the newest N - H samples of the stream become the next call's overlap
        const long a_end = (p.first_hop + f_end) * (long) H;
        float* to = p.tail_out + track * (long) (N - H);
        for (int i = t; i < N - H; i += T) to[i] = sm.ring[sk32 ((int) ((a_end - (N - H) + i) & (N - 1)))];
    }
}

// ---------------------------------------------------------------------------------------------------------
// K1b: the scalar tail of both analyser bodies, one thread per frame, one warp per batch of 32 consecutive frames.
// A batch's records are one contiguous run of 32 * frame_rec_bytes (9.5 .. 24.5 KB): it arrives in shared memory by ONE
// bulk copy (a thread reading its own 304 .. 784-byte record straight from global memory touches a different sector with
// every load).  The tail is a long dependent fp64 chain (pow, five log10, three sqrt), so it needs many resident warps, and
// the staged records would cap them: a block of 12 warps therefore shares THREE staging buffers in turn.  Warp w waits for
// its batch in buffer w % 3, reduces the per-warp partials of its 32 frames into registers, hands the buffer to batch
// w + 3 (it issues that copy itself: no "buffer empty" barrier) and runs the tail while the later batches stream in.
constexpr int kFzWarps = 12, kFzBufs = 3, kFzBlocks = 2;
constexpr int kFinalizeRows = 32 * kFzWarps;
template <int NW>
__global__ void __launch_bounds__ (kFinalizeRows, kFzBlocks) k_finalize (const FinalizeParams p)
{
    constexpr size_t RB = sizeof (FrameHead) + NW * sizeof (WarpPart);
    constexpr size_t BB = 32 * RB;
    extern __shared__ __align__ (128) unsigned char fz_smem[];            // [kFzBufs][BB]
    __shared__ uint64_t fz_full[kFzWarps];                              // one per batch, each completes once (a waiter may lag one phase at most)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long row0 = (long) blockIdx.x * kFinalizeRows;
    auto batch_rows = [&] (int batch) -> int
    {
        const long left = p.n_rows - (row0 + 32L * batch);
        return batch < kFzWarps ? (int) (left < 0 ? 0 : (left > 32 ? 32 : left)) : 0;
    };
    auto issue = [&] (int batch)                                          // one lane: start the copy of a batch's records
    {
        const int rows = batch_rows (batch);
        if (rows <= 0) return;
        uint64_t* bar = &fz_full[batch];
        mbar_expect_tx (bar, (uint32_t) (rows * RB));
        bulk_g2s (fz_smem + (batch % kFzBufs) * BB, p.rec + (size_t) (row0 + 32L * batch) * RB, (uint32_t) (rows * RB), bar);
    };
    if (threadIdx.x == 0)
    {
        for (int b = 0; b < kFzWarps; ++b) mbar_init (&fz_full[b], 1);
        asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp < kFzBufs && lane == 0) issue (warp);
    const int rows = batch_rows (warp);
    if (rows <= 0) return;                                                // (whole warp: the later batches are empty as well)
    mbar_wait (&fz_full[warp], 0u);
    const unsigned char* mine = fz_smem + (warp % kFzBufs) * BB + (size_t) lane * RB;     // lanes >= rows read stale bytes and leave below
    const FrameHead r = *reinterpret_cast<const FrameHead*> (mine);
    const WarpPart* rw = reinterpret_cast<const WarpPart*> (mine + sizeof (FrameHead));
    const long idx = row0 + 32L * warp + lane;
    float* out = p.raw + idx * FX_NUM_FEATURES;
    const int N = p.window, M = N / 2;                            // NW = N / 512 warps of the K1 CTA left the partials
    const double nyquist = p.sample_rate / 2.0;

    // ---- the per-warp partials, added over the warps as a pairwise tree (the order of a butterfly over the warps) ------
    // (value by value, so that at most NW partials are live at a time)
    auto tree = [&] (auto get) -> double
    {
        double v[NW];
        #pragma unroll
        for (int w = 0; w < NW; ++w) v[w] = get (w);
        #pragma unroll
        for (int half = 1; half < NW; half <<= 1)
            #pragma unroll
            for (int w = 0; w < NW; w += 2 * half) v[w] += v[w + half];
        return v[0];
    };
    const double w1 = tree ([&] (int w) { return rw[w].p1d[1]; }), s2 = tree ([&] (int w) { return rw[w].p1d[2]; });
    const double s4 = tree ([&] (int w) { return rw[w].p1d[3]; }), flux = tree ([&] (int w) { return rw[w].p1f[0]; });
    const double lhr = tree ([&] (int w) { return rw[w].p1f[1]; }), flat_sum = tree ([&] (int w) { return rw[w].p1f[2]; });
    const double inharm = tree ([&] (int w) { return rw[w].inharm; });
    int count_i = 0, npeaks_i = 0;
    float rawmax = 0.0f;
    #pragma unroll
    for (int w = 0; w < NW; ++w) { count_i += rw[w].count; npeaks_i += rw[w].npeaks; rawmax = fmaxf (rawmax, rw[w].rawmax); }
    ME tot[NW];
    #pragma unroll
    for (int w = 0; w < NW; ++w) { tot[w].m = rw[w].scan_m; tot[w].e = rw[w].scan_e; }
    // every value of the batch is in registers: the buffer goes to batch warp + kFzBufs
    __syncwarp();
    if (lane == 0 && batch_rows (warp + kFzBufs) > 0) { fence_proxy_async(); issue (warp + kFzBufs); }
    if (lane >= rows) return;

    const double count = (double) count_i;
    const double max_e = fmax ((double) rawmax, r.maxmag);                                        // SpectralCharacteristics.h:153-163
    // flatness product (:89-94): K1 reports a range event with the replayed product; otherwise the product of the warps' totals
    double product = r.product; float flat_state = r.flat_state;
    if (flat_state < 0.0f)
    {
        #pragma unroll
        for (int half = 1; half < NW; half <<= 1)
            #pragma unroll
            for (int w = 0; w < NW; w += 2 * half) tot[w] = me_mul (tot[w], tot[w + half]);
        product = ldexp_normal (tot[0].m, tot[0].e);
        flat_state = 0.0f;
    }

    // ---- spectral body (SpectralCharacteristics.h:100-143, :145-200) ------------------------------------------
    const float rms = (float) sqrt (r.rms_sum / (double) N);                                      // getRMSLevel
    const float log_rms = (float) log10 ((double) __fadd_rn (__fmul_rn (rms, 9.0f), 1.0f));       // RealTimeAnalyser.h:208
    const double eps = 0.01 * (double) log_rms;                                                   // :108
    const bool silent = ! (r.mag_sum > 0.05);                                                     // :121-123
    // K1 leaves raw moments over x = (bin + 1/2) / M = fc / nyquist: W1 = sum x mag, S2 = sum x^2 mag, S4 = sum mag^2
    // (see the top of this file)
    const float  centroid = (float) ((w1 * nyquist) / r.mag_sum);                                 // :127 weighted / magSum
    const double cn = (double) centroid / nyquist;                                                // :137
    const double var = (s2 - 2.0 * cn * w1) + cn * cn * r.mag_sum;                                // :135-139
    const double inv_max_e = 1.0 / max_e;
    const double mean_e = (r.mag_sum * inv_max_e) / (double) M;                                   // :177
    const double sie = ((double) M * w1 - 0.5 * r.mag_sum) * inv_max_e;                           // :175 sum i e_i
    double evar = s4 * inv_max_e * inv_max_e - (double) M * mean_e * mean_e;                      // :182-190
    if (evar < 0.0) evar = 0.0;                                   // rounding of the difference (a spectrum flat to ~1e-8)
    float gate_margin = fminf (relmargin_d (r.mag_sum, 0.05), relmargin_d (max_e, 0.0001));
    float o_centroid = 0.0f, o_spread = 0.0f, o_flat = 0.0f, o_ler = 0.0f, o_flux = 0.0f, o_slope = 0.0f;
    if (! silent)
    {
        const float max_flux = (float) (M * (M + 1)) / 2.0f;                                      // :111
        const double inv = 1.0 / (count > 0.0 ? count : 1.0);                                 // :130
        const float flat = flat_sum > eps ? (float) (pow (product, inv) / (inv * flat_sum)) : 0.0f;     // :57-60
        o_flat = (float) log10 ((double) flat * 9.0 + 1.0);                                       // :132
        const float c = __fdiv_rn (centroid, (float) (nyquist / 2.0));                            // :133
        o_centroid = (float) log10 ((double) __fadd_rn (__fmul_rn (c, 9.0f), 1.0f));              // :134
        const float max_spread = (float) (((double) centroid / nyquist) * (1.0 - ((double) centroid / nyquist)));   // :140
        o_spread = (float) ((var / r.mag_sum) / (double) max_spread);                             // :141
        o_ler = (float) (lhr / r.mag_sum);                                                      // :125
        o_flux = r.have_prev != 0.0f ? (float) (flux / (double) max_flux) : 0.0f;               // :112 (K2 fixes the chunk's first non-silent frame)
    }
    if (max_e > 0.0001)                                                                         // :165-167
    {
        const double energy_var = evar / (double) M;
        const double bin_std = sqrt (p.bin_var), energy_std = sqrt (energy_var);
        const double rr = (sie - ((double) M * mean_e * 0.5)) / (double) ((float) M - 1.0f) * energy_std * bin_std;   // :195
        o_slope = (float) (rr * (bin_std / energy_std));                                          // :198
    }

    // ---- harmonic body (PitchAnalyser.h:57, RealTimeAnalyser.h:165-172, HarmonicCharacteristics.h:88-105) ---------
    const double f0 = (nyquist * 2.0) / (double) r.lag;
    float o_her = 0.0f, o_oer = 0.0f, o_inh = 0.0f;
    if (! (r.hsum < 0.005))
    {
        // calculateHarmonicEnergyCharacteristics (:147-198): 15 sub-octave terms, then the harmonics 1..3; each term is the
        // normalised magnitude (float) (mag / max) (:75-76) of the largest |Re A| K1 found around its bin (< 0: term not used)
        double score = 0.0, even = 0.0, odd = 0.0;
        #pragma unroll
        for (int l = 0; l < 18; ++l)
        {
            const float mx = r.her_mx[l];
            const double term = mx < 0.0f ? 0.0 : (double) (float) (((double) mx * (double) mx) / r.hmax);
            score += term;
            if (l == 16) even = term;                                                             // harmonic 2
            if (l == 15 || l == 17) odd += term;                                                  // harmonics 1 and 3
        }
        // the normalised magnitudes (:71-77) sum to magnitudeSum / maxMagnitude up to fp64 rounding
        double her = score / (r.hsum / r.hmax);                                                   // :186-188
        her = her > 1.0 ? 1.0 : her; her = her < 0.0 ? 0.0 : her;
        double oer = 1.0;
        if (odd > 0.0) oer = even / odd;                                                          // :190-195
        oer = oer > 1.0 ? 1.0 : oer; oer = oer < 0.0 ? 0.0 : oer;
        o_her = (float) log10 ((double) (float) her * 9.0 + 1.0);                                 // :101-103
        o_oer = (float) log10 ((double) (float) oer * 9.0 + 1.0);
        // :237 (K1 leaves the sum of f0Proportion * binMagnitude; with no contributing peak the reference's sum stays 0 whatever
        // the magnitude sum is -- NaN input included)
        o_inh = (float) log10 ((inharm != 0.0 ? inharm / r.hsum : 0.0) * 9.0 + 1.0);
    }
    gate_margin = fminf (gate_margin, relmargin_d (r.hsum, 0.005));

    out[FX_ONSET] = 0.0f;
    out[FX_RMS] = log_rms;
    out[FX_F0] = (float) (f0 / 5000.0);
    out[FX_CENTROID] = o_centroid; out[FX_SPREAD] = o_spread; out[FX_FLATNESS] = o_flat;
    out[FX_LER] = o_ler; out[FX_FLUX] = o_flux; out[FX_SLOPE] = o_slope;
    out[FX_HER] = o_her;
    out[FX_OER] = o_her;                                                                          // RealTimeAnalyser.h:171 stores HER in the OER slot
    out[FX_INHARM] = o_inh;
    if (p.diag)
    {
        float* dg = p.diag + idx * FX_NUM_DIAG;
        dg[FX_DIAG_TRUE_OER] = o_oer;
        dg[FX_DIAG_LAG] = r.lag;
        dg[FX_DIAG_PITCH_MARGIN] = r.pitch_margin;
        dg[FX_DIAG_NUM_PEAKS] = r.hsum < 0.005 ? 0.0f : (float) npeaks_i;                           // HarmonicCharacteristics.h:88
        dg[FX_DIAG_PEAK_MARGIN] = r.peak_margin;
        dg[FX_DIAG_FLAT_COUNT] = (float) count;
        // The gate compares Re^2 with eps; Re carries the absolute rounding noise of an fp32 FFT (here and in the reference's
        // own transform), taken as 1e-6 of the spectrum's rms like the pitch margin's floor.  For every bin the relative gap
        // shrinks by at most 2 e / sqrt (eps) + e^2 / eps (|Re| >= sqrt (eps) above the gate, the gap is relative to eps below).
        float fm = r.flat_margin;
        if (eps > 0.0)
        {
            const double e_abs = 1.0e-6 * sqrt (r.mag_sum / (double) M);
            fm = fmaxf (0.0f, fm - (float) (2.0 * e_abs / sqrt (eps) + e_abs * e_abs / eps));
        }
        dg[FX_DIAG_FLAT_MARGIN] = fm;
        dg[FX_DIAG_GATE_MARGIN] = gate_margin;
        dg[FX_DIAG_ONSET_MARGIN] = 1.0f;
        dg[FX_DIAG_FLAT_STATE] = flat_state;
    }
}

// ---------------------------------------------------------------------------------------------------------
template <int R1, bool SO> static void launch_so (unsigned g, const AnalyseParams& p, cudaStream_t stream)
{
    const unsigned nt = 16 * R1;
    const size_t smem = sizeof (Smem<R1>);
    if (p.spectrum == FX_SPECTRUM_POWER)
    {
        if (p.want_margins) k_analyse<R1, true, true, SO><<<g, nt, smem, stream>>> (p);
        else                k_analyse<R1, false, true, SO><<<g, nt, smem, stream>>> (p);
    }
    else
    {
        if (p.want_margins) k_analyse<R1, true, false, SO><<<g, nt, smem, stream>>> (p);
        else                k_analyse<R1, false, false, SO><<<g, nt, smem, stream>>> (p);
    }
}

template <int R1> static cudaError_t launch_t (long n_tracks, const AnalyseParams& p, cudaStream_t stream)
{
    const long grid = n_tracks * p.n_chunks;
    if (grid <= 0) return cudaSuccess;
    if (p.spec) launch_so<R1, true> ((unsigned) grid, p, stream);
    else        launch_so<R1, false> ((unsigned) grid, p, stream);
    return cudaGetLastError();
}

template <int R1, bool SO> static cudaError_t configure_so()
{
    const int smem = (int) sizeof (Smem<R1>);
    cudaError_t ce = cudaFuncSetAttribute (k_analyse<R1, true, false, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute (k_analyse<R1, false, false, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute (k_analyse<R1, true, true, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute (k_analyse<R1, false, true, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return ce;
}

template <int R1> static cudaError_t configure_t()
{
    cudaError_t ce = cudaFuncSetAttribute (k_finalize<R1 / 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (kFzBufs * 32 * frame_rec_bytes (256 * R1)));
    if (ce == cudaSuccess) ce = configure_so<R1, false>();
    if (ce == cudaSuccess) ce = configure_so<R1, true>();
    return ce;
}

int analyse_ctas_per_sm (int window)
{
    return window == 4096 ? kCtasR16 : (window == 2048 ? kCtasR8 : kCtasR4);
}

size_t analyse_smem_bytes (int window)
{
    switch (window)
    {
        case 1024: return sizeof (Smem<4>);
        case 2048: return sizeof (Smem<8>);
        case 4096: return sizeof (Smem<16>);
        default:   return 0;
    }
}

cudaError_t configure_analyse (int window)
{
    switch (window)
    {
        case 1024: return configure_t<4>();
        case 2048: return configure_t<8>();
        case 4096: return configure_t<16>();
        default:   return cudaErrorInvalidValue;
    }
}

cudaError_t launch_analyse (int window, long n_tracks, const AnalyseParams& p, cudaStream_t stream)
{
    switch (window)
    {
        case 1024: return launch_t<4>  (n_tracks, p, stream);
        case 2048: return launch_t<8>  (n_tracks, p, stream);
        case 4096: return launch_t<16> (n_tracks, p, stream);
        default:   return cudaErrorInvalidValue;
    }
}

cudaError_t launch_finalize (const FinalizeParams& p, cudaStream_t stream)
{
    if (p.n_rows <= 0) return cudaSuccess;
    const unsigned grid = (unsigned) ((p.n_rows + kFinalizeRows - 1) / kFinalizeRows);
    const size_t smem = (size_t) kFzBufs * 32 * frame_rec_bytes (p.window);
    switch (p.window)
    {
        case 1024: k_finalize<2><<<grid, kFinalizeRows, smem, stream>>> (p); break;
        case 2048: k_finalize<4><<<grid, kFinalizeRows, smem, stream>>> (p); break;
        case 4096: k_finalize<8><<<grid, kFinalizeRows, smem, stream>>> (p); break;
        default:   return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

} // namespace fx

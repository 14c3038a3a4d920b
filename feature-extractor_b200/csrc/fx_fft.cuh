// fx_fft.cuh -- shared-memory N-point complex FFT for one CTA (sm_100a), N = R1 * 16 * 16,
// R1 in {4, 8, 16}  ->  N in {1024, 2048, 4096}, T = N / 16 threads, 16 complex points per thread.
//
// Replaces juce::FFT as reached through RealTimeFFT (Source/RealTimeAudioAnalysis.h:159-189).
//
// Decimation in frequency, three register-resident stages (radix R1, 16, 16) with two exchanges
// through shared memory:
//   n = n1 * 256 + m            (m = n2 * 16 + n3)        k = k1 + R1 * k2 + 16 * R1 * k3
//   stage 1: butterfly m   : R1-point DFT over n1, twiddle W_N^(m k1)     -> ex[k1][m]
//   stage 2: (k1, n3)      : 16-point DFT over n2, twiddle W_256^(n3 k2)  -> ex[k1][k2][n3]   (in place)
//   stage 3: (k1, k2)      : 16-point DFT over n3                         -> ex[k1][k2][k3]   (in place)
// Every stage is in place per thread, and the 16 threads that share a row k1 in stages 2 and 3 are one half warp, so the
// only block-wide barrier inside a transform is the one between stage 1 and stage 2; the 2 -> 3 exchange needs a
// __syncwarp.  The spectrum is left in "digit order": X[k], k = k1 + R1 k2 + 16 R1 k3, lives at zpos (k) =
// k1 * ROW + 17 k2 + k3, and the time samples a transform starts from at tpos (n) = (n >> 8) * ROW + phys (n & 255).
// Rows are 273 elements apart and 16-element groups inside a row are skewed by one (phys (a) = a + (a >> 4)): the row
// accesses of stage 2, the column accesses of stage 3 and the readers of runs of consecutive bins are conflict free.
// Twiddles come from tables evaluated in double on the host and rounded to fp32 (as JUCE does).  The stage-1 twiddles
// W_N^(m k1) are read from a full global table through L1 (one 8-byte load per twiddle: 1.7 % faster than forming each one
// from two small shared-memory factors); that table holds the fp32 products of the two factors, rounded as the in-line
// product was (fx_tables.cu).
//
// Twiddle powers: only the twiddles W^1, W^2, W^4, W^8 of a thread are loaded (exact table values); the other eleven are
// products of those, at most three multiplications deep (W^15 = W^8 W^4 W^2 W^1): 11 packed complex multiplies in place of 11
// loads per stage and transform.  The loads ride the L1 / shared-memory data pipe, the busiest unit of the kernel, and the
// stage-1 ones (global table through L1) expose their latency.  Measured (profiles/r02_v22_ab_*.txt), kernel ms at
// N = 4096 / 2048 / 1024:  all loads 68.43 / 33.11 / 34.11;  stage 1 by powers 66.16 / 32.78 / 34.11;  stage 2 by powers
// 68.14 / 33.51 / 34.23;  both 65.84 / 33.25 / 33.84.  K1 takes both stages by powers at every size (fx_analyse.cu).
#pragma once
#include <cuda_runtime.h>

namespace fx {

__device__ __forceinline__ int phys (int a) { return a + (a >> 4); }

// Packed fp32 arithmetic (sm_100a FADD2 / FMUL2 / FFMA2): one instruction works on both halves of a 64-bit register
// pair, IEEE round-to-nearest per half like the scalar forms.  A complex value is such a pair, so a complex add is one
// instruction and a complex multiply two; ptxas folds the component swaps and negations of the operands below into
// the instructions' operand modifiers (.LO_HI, .NP, .F32 broadcast).  The kernel is bound by issue slots, not by the
// FP32 pipe: the packed forms halve the issue slots of the butterflies.
__device__ __forceinline__ float2 f2add (float2 a, float2 b)
{
    float2 r;
    asm ("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0, %1}, rc;}"
         : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 f2sub (float2 a, float2 b)
{
    float2 r;
    asm ("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; sub.rn.f32x2 rc, ra, rb; mov.b64 {%0, %1}, rc;}"
         : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 f2mul (float2 a, float2 b)
{
    float2 r;
    asm ("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mul.rn.f32x2 rc, ra, rb; mov.b64 {%0, %1}, rc;}"
         : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 f2fma (float2 a, float2 b, float2 c)
{
    float2 r;
    asm ("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mov.b64 rc, {%6, %7}; fma.rn.f32x2 rd, ra, rb, rc; mov.b64 {%0, %1}, rd;}"
         : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return r;
}

__device__ __forceinline__ float2 cadd (float2 a, float2 b) { return f2add (a, b); }
__device__ __forceinline__ float2 csub (float2 a, float2 b) { return f2sub (a, b); }

// a * w (forward) or a * conj (w) (inverse): (a.x w.x -+ a.y w.y, a.y w.x +- a.x w.y) as one packed multiply and one packed FMA
template <bool INV>
__device__ __forceinline__ float2 cmulw (float2 a, float2 w)
{
    const float2 wy = make_float2 (w.y, w.y), wx = make_float2 (w.x, w.x);
    if (INV) return f2fma (a, wx, f2mul (make_float2 (a.y, -a.x), wy));
    else     return f2fma (a, wx, f2mul (make_float2 (-a.y, a.x), wy));
}

// multiply by -i (forward) / +i (inverse)
template <bool INV>
__device__ __forceinline__ float2 mul_mi (float2 a)
{
    if (INV) return make_float2 (-a.y, a.x);
    else     return make_float2 (a.y, -a.x);
}

template <bool INV>
__device__ __forceinline__ void radix2 (float2& a0, float2& a1)
{
    const float2 t = a0;
    a0 = cadd (t, a1);
    a1 = csub (t, a1);
}

// 4-point DFT in place: slot j <- X[j]
template <bool INV>
__device__ __forceinline__ void radix4 (float2& a0, float2& a1, float2& a2, float2& a3)
{
    const float2 t0 = cadd (a0, a2), t1 = csub (a0, a2);
    const float2 t2 = cadd (a1, a3), t3 = mul_mi<INV> (csub (a1, a3));
    a0 = cadd (t0, t2);
    a2 = csub (t0, t2);
    a1 = cadd (t1, t3);
    a3 = csub (t1, t3);
}

#define FX_C1 0.92387953251128675613f   /* cos (pi / 8) */
#define FX_S1 0.38268343236508977173f   /* sin (pi / 8) */
#define FX_R2 0.70710678118654752440f   /* sqrt (1/2)  */

// R-point DFT in registers; afterwards slot s holds X[out_index<R> (s)].
template <int R> __device__ __forceinline__ constexpr int out_index (int s)
{
    return R == 16 ? ((s >> 2) + 4 * (s & 3)) : (R == 8 ? ((s >> 2) + 2 * (s & 3)) : s);
}
// inverse of out_index: the slot that holds X[k]
template <int R> __device__ __forceinline__ constexpr int slot_of (int k)
{
    return R == 16 ? ((k >> 2) + 4 * (k & 3)) : (R == 8 ? ((k >> 1) + 4 * (k & 1)) : k);
}

template <int R, bool INV>
__device__ __forceinline__ void butterfly (float2* v)
{
    if (R == 16)
    {
        #pragma unroll
        for (int n0 = 0; n0 < 4; ++n0) radix4<INV> (v[n0], v[n0 + 4], v[n0 + 8], v[n0 + 12]);
        // slot n0 + 4 ka *= W16^(n0 ka)
        v[5]  = cmulw<INV> (v[5],  make_float2 ( FX_C1, -FX_S1));   // e = 1
        v[6]  = cmulw<INV> (v[6],  make_float2 ( FX_R2, -FX_R2));   // e = 2
        v[7]  = cmulw<INV> (v[7],  make_float2 ( FX_S1, -FX_C1));   // e = 3
        v[9]  = cmulw<INV> (v[9],  make_float2 ( FX_R2, -FX_R2));   // e = 2
        v[10] = mul_mi<INV> (v[10]);                                // e = 4
        v[11] = cmulw<INV> (v[11], make_float2 (-FX_R2, -FX_R2));   // e = 6
        v[13] = cmulw<INV> (v[13], make_float2 ( FX_S1, -FX_C1));   // e = 3
        v[14] = cmulw<INV> (v[14], make_float2 (-FX_R2, -FX_R2));   // e = 6
        v[15] = cmulw<INV> (v[15], make_float2 (-FX_C1,  FX_S1));   // e = 9
        #pragma unroll
        for (int ka = 0; ka < 4; ++ka) radix4<INV> (v[4 * ka], v[4 * ka + 1], v[4 * ka + 2], v[4 * ka + 3]);
    }
    else if (R == 8)
    {
        #pragma unroll
        for (int n0 = 0; n0 < 4; ++n0) radix2<INV> (v[n0], v[n0 + 4]);
        v[5] = cmulw<INV> (v[5], make_float2 ( FX_R2, -FX_R2));
        v[6] = mul_mi<INV> (v[6]);
        v[7] = cmulw<INV> (v[7], make_float2 (-FX_R2, -FX_R2));
        radix4<INV> (v[0], v[1], v[2], v[3]);
        radix4<INV> (v[4], v[5], v[6], v[7]);
    }
    else
    {
        radix4<INV> (v[0], v[1], v[2], v[3]);
    }
}

// w[k] = w1^k for k = 1 .. R - 1 from the exact values of w1^1, w1^2, w1^4, w1^8 (slots 1, 2, 4, 8 filled by the caller)
template <int R>
__device__ __forceinline__ void twiddle_powers (float2* w)
{
    w[3] = cmulw<false> (w[2], w[1]);
    if (R > 4)
    {
        w[5] = cmulw<false> (w[4], w[1]); w[6] = cmulw<false> (w[4], w[2]); w[7] = cmulw<false> (w[4], w[3]);
    }
    if (R > 8)
    {
        w[9]  = cmulw<false> (w[8], w[1]); w[10] = cmulw<false> (w[8], w[2]); w[11] = cmulw<false> (w[8], w[3]);
        w[12] = cmulw<false> (w[8], w[4]); w[13] = cmulw<false> (w[8], w[5]); w[14] = cmulw<false> (w[8], w[6]);
        w[15] = cmulw<false> (w[8], w[7]);
    }
}

// the powers above R / 2 that twiddle_powers<R> forms and twiddle_powers<R / 2> does not (w[3] .. w[R/2] already filled)
template <int R>
__device__ __forceinline__ void twiddle_powers_upper (float2* w)
{
    if (R == 4) w[3] = cmulw<false> (w[2], w[1]);
    if (R == 8) { w[5] = cmulw<false> (w[4], w[1]); w[6] = cmulw<false> (w[4], w[2]); w[7] = cmulw<false> (w[4], w[3]); }
    if (R == 16)
    {
        w[9]  = cmulw<false> (w[8], w[1]); w[10] = cmulw<false> (w[8], w[2]); w[11] = cmulw<false> (w[8], w[3]);
        w[12] = cmulw<false> (w[8], w[4]); w[13] = cmulw<false> (w[8], w[5]); w[14] = cmulw<false> (w[8], w[6]);
        w[15] = cmulw<false> (w[8], w[7]);
    }
}

// Shared-memory footprint helpers (in elements)
template <int R1> struct FftDims
{
    static constexpr int N       = R1 * 256;
    static constexpr int T       = R1 * 16;            // threads
    static constexpr int Q1      = 16 / R1;            // stage-1 butterflies per thread
    static constexpr int ROW     = 273;                // 256 * 17 / 16 + 1: consecutive bins (consecutive k1) fall into different banks
    static constexpr int EX_LEN  = R1 * ROW;           // float2 elements in the exchange buffer
    static constexpr int TW2_FULL = 15 * 16;           // float2, tw2[(k2 - 1) * 16 + n3]      = W_256^(n3 k2)
    // stage-2 twiddles by powers: the shared-memory copy holds only the rows k2 = 1, 2, 4, 8 (in that order), and it lives in
    // the 16-byte holes of the caller's skewed sample ring (fx_analyse.cu: one unused float4 behind every 32 floats): element
    // e = row * 16 + n3 sits in hole e / 2, slot e % 2, holes 36 floats = 18 float2 apart.  The 16 lanes of a half warp read
    // 8 holes, i.e. 8 different 16-byte bank groups: conflict free like the dense table.
    static constexpr int TW2_HOLE_ROW = 8 * 18;        // float2 distance between the rows k2 = 1, 2, 4, 8 of one n3
};

// Stage 1 on v (slot q * R1 + n1 = input n1 of butterfly q), then twiddle and store to ex.
// PRUNABLE: a runtime flag even says that the input is even (z[(N - n) & (N - 1)] = z[n], real and imaginary parts alike), so
// X[N - k] = X[k] and row R1 - k1 of the exchange buffer holds the mirrors of row k1.  Outputs k1 > R1 / 2 are then neither
// twiddled nor stored, and with them go the twiddle powers above R1 / 2, which only those rows use; the caller skips stages 2
// and 3 of those rows.  The flag is uniform, so this is one branch per butterfly.
template <int R1, bool INV, bool PRUNABLE = false>
__device__ __forceinline__ void fft_stage1_store (float2* v, int m0, float2* __restrict__ ex, const float2* __restrict__ tw1f, bool even = false)
{
    using D = FftDims<R1>;
    #pragma unroll
    for (int q = 0; q < D::Q1; ++q)
    {
        butterfly<R1, INV> (v + q * R1);
        const int m = m0 + D::T * q;
        const int pm = phys (m);
        float2 wp[16];
        wp[1] = __ldg (&tw1f[m]); wp[2] = __ldg (&tw1f[256 + m]);
        if (R1 > 4) wp[4] = __ldg (&tw1f[3 * 256 + m]);
        if (R1 > 8) wp[8] = __ldg (&tw1f[7 * 256 + m]);
        if (! PRUNABLE)
        {
            twiddle_powers<R1> (wp);
            #pragma unroll
            for (int s = 0; s < R1; ++s)
            {
                const int k1 = out_index<R1> (s);
                float2 val = v[q * R1 + s];
                if (k1 > 0) val = cmulw<INV> (val, wp[k1]);
                ex[k1 * D::ROW + pm] = val;
            }
            continue;
        }
        twiddle_powers<R1 / 2> (wp);
        #pragma unroll
        for (int s = 0; s < R1; ++s)
        {
            const int k1 = out_index<R1> (s);
            if (k1 > R1 / 2) continue;
            float2 val = v[q * R1 + s];
            if (k1 > 0) val = cmulw<INV> (val, wp[k1]);
            ex[k1 * D::ROW + pm] = val;
        }
        if (! even)
        {
            twiddle_powers_upper<R1> (wp);
            #pragma unroll
            for (int s = 0; s < R1; ++s)
            {
                const int k1 = out_index<R1> (s);
                if (k1 <= R1 / 2) continue;
                ex[k1 * D::ROW + pm] = cmulw<INV> (v[q * R1 + s], wp[k1]);
            }
        }
    }
}

// Stage 2 in place (one 16-point butterfly per thread).  Caller syncs before and after.  POWERS: tw2 is the compact table
// in the holes of the ring (see FftDims), else the full table tw2[(k2 - 1) * 16 + n3].
template <int R1, bool INV, bool POWERS>
__device__ __forceinline__ void fft_stage2 (int t, float2* __restrict__ ex, const float2* __restrict__ tw2)
{
    using D = FftDims<R1>;
    const int k1 = t >> 4, n3 = t & 15;
    float2* row = ex + k1 * D::ROW + n3;
    float2 v[16];
    #pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) v[n2] = row[n2 * 17];
    butterfly<16, INV> (v);
    float2 wp[16];
    if (POWERS)
    {
        const float2* th = tw2 + 18 * (n3 >> 1) + (n3 & 1);                                  // tw2: first hole of the ring
        wp[1] = th[0]; wp[2] = th[D::TW2_HOLE_ROW]; wp[4] = th[2 * D::TW2_HOLE_ROW]; wp[8] = th[3 * D::TW2_HOLE_ROW];
        twiddle_powers<16> (wp);
    }
    #pragma unroll
    for (int s = 0; s < 16; ++s)
    {
        const int k2 = out_index<16> (s);
        float2 val = v[s];
        if (k2 > 0) val = cmulw<INV> (val, POWERS ? wp[k2] : tw2[(k2 - 1) * 16 + n3]);
        row[k2 * 17] = val;
    }
}

// Stage 3 in place: X[k1 + R1 k2 + 16 R1 k3] replaces element (k2, n3 = k3) of row k1.  The caller has made the stage-2
// stores of this half warp visible (__syncwarp).  rowmask: the lanes that run this stage together (at least the half warp
// of the row; a caller whose other half warp skips the stage passes the half warp alone).
template <int R1, bool INV>
__device__ __forceinline__ void fft_stage3 (int t, float2* __restrict__ ex, unsigned rowmask = 0xffffffffu)
{
    using D = FftDims<R1>;
    const int k1 = t >> 4, k2 = t & 15;
    float2* col = ex + k1 * D::ROW + k2 * 17;
    float2 v[16];
    #pragma unroll
    for (int n3 = 0; n3 < 16; ++n3) v[n3] = col[n3];
    butterfly<16, INV> (v);
    __syncwarp (rowmask);                                 // every thread of the row has read its column
    #pragma unroll
    for (int s = 0; s < 16; ++s) col[out_index<16> (s)] = v[s];
}

// position of spectrum bin k / of time sample n in the exchange buffer (see the header comment)
template <int R1> __device__ __forceinline__ int zpos (int k)
{
    using D = FftDims<R1>;
    return (k & (R1 - 1)) * D::ROW + ((k / R1) & 15) * 17 + k / (16 * R1);
}
template <int R1> __device__ __forceinline__ int tpos (int n)
{
    return (n >> 8) * FftDims<R1>::ROW + phys (n & 255);
}
// zpos (b + j) - zpos (b) for a run of bins that starts at a multiple of 8 (j < 8) or of 16 (j < 16): a compile-time offset
template <int R1> __device__ __forceinline__ constexpr int zrun (int j)
{
    return (j & (R1 - 1)) * FftDims<R1>::ROW + (j / R1) * 17;
}

} // namespace fx

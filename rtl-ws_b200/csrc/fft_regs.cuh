// fft_regs.cuh -- fully unrolled in-register forward FFTs (radix-2 DIT with FMA-fused
// butterflies, sizes 2..64) on PACKED complex numbers: one 64-bit register pair holds (re, im) and every butterfly is a
// Blackwell f32x2 instruction (FADD2 / FMUL2 / FFMA2, sm_100 PTX add/mul/fma.rn.f32x2).
//
// Why packed: the FP32 pipe retires 128 lanes/clk/SM either way (tools/ubench.cu measures
// 125 scalar vs 128 packed results/clk/SM on B200), but a packed instruction carries two
// results per ISSUE slot, and the spectrum kernel is issue-bound (profiles/).  The lane
// swap and per-lane negation that complex arithmetic needs (multiply by -i, the cross terms
// of a complex product) are operand modifiers in SASS (R.F32x2.LO_HI, .NP), so they cost
// nothing: ptxas folds the mov.b64 shuffles below into the consuming instruction.
//
// One thread owns R complex points.  All twiddles inside a size-R transform are
// compile-time constants (multiples of 2*pi/64).  Input is taken in bit-reversed register
// order and output is natural; callers permute by renaming registers (bitrev<R>() is
// constexpr), which is free.
//
// Sign convention: X[k] = sum_j x[j] exp(-2*pi*i*j*k/R)  -- the FFTW_FORWARD transform the
// reference plans at spectrum.c:42.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

typedef unsigned long long c64;      // packed complex: low word = re, high word = im

__device__ __forceinline__ c64 cpack(float re, float im)
{
    c64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(re), "f"(im));
    return r;
}
__device__ __forceinline__ void cunpack(c64 v, float& re, float& im)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(re), "=f"(im) : "l"(v));
}
__device__ __forceinline__ c64 cadd(c64 a, c64 b)
{
    c64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ c64 csub(c64 a, c64 b)
{
    c64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ c64 cmul2(c64 a, c64 b)      // lane-wise product
{
    c64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ c64 cfma2(c64 a, c64 b, c64 c)   // lane-wise a * b + c
{
    c64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// Store a packed complex number.  Written as two float halves on purpose: with a 64-bit store of the
// packed register ptxas first copies every value that was also unpacked somewhere (the "2u - s" form of
// the butterflies unpacks s) into a scratch register pair -- one MOV pair per stored value.
__device__ __forceinline__ void cstore(c64* dst, c64 v)
{
    float re, im;
    cunpack(v, re, im);
    *reinterpret_cast<float2*>(dst) = make_float2(re, im);
}
// general complex product a * w with w = (wr, wi):  (ar*wr - ai*wi, ai*wr + ar*wi)
//   = a * (wr, wr) + (-ai, ar) * (wi, wi)
__device__ __forceinline__ c64 cmul(c64 a, float wr, float wi)
{
    float ar, ai;
    cunpack(a, ar, ai);
    return cfma2(a, cpack(wr, wr), cmul2(cpack(-ai, ar), cpack(wi, wi)));
}

// cos(2*pi*q/32), q = 0..8 (first octant + quadrant end)
__host__ __device__ constexpr float cos32_table(int q)
{
    return q == 0   ? 1.0f
           : q == 1 ? 0.98078528040323044913f
           : q == 2 ? 0.92387953251128675613f
           : q == 3 ? 0.83146961230254523708f
           : q == 4 ? 0.70710678118654752440f
           : q == 5 ? 0.55557023301960222474f
           : q == 6 ? 0.38268343236508977173f
           : q == 7 ? 0.19509032201612826785f
                    : 0.0f;
}

// cos / sin of 2*pi*q/32 for any integer q
__host__ __device__ constexpr float cos32(int q)
{
    q &= 31;
    if (q > 16) q = 32 - q;                 // cos is even about pi
    return q <= 8 ? cos32_table(q) : -cos32_table(16 - q);
}
__host__ __device__ constexpr float sin32(int q)
{
    return cos32(q - 8);
}

// cos(2*pi*q/64), q = 0..16, for the 64-point transform of the four-step kernel
__host__ __device__ constexpr float cos64_table(int q)
{
    return q == 0    ? 1.0f
           : q == 1  ? 0.99518472667219688624f
           : q == 2  ? 0.98078528040323044913f
           : q == 3  ? 0.95694033573220886494f
           : q == 4  ? 0.92387953251128675613f
           : q == 5  ? 0.88192126434835502971f
           : q == 6  ? 0.83146961230254523708f
           : q == 7  ? 0.77301045336273696081f
           : q == 8  ? 0.70710678118654752440f
           : q == 9  ? 0.63439328416364549822f
           : q == 10 ? 0.55557023301960222474f
           : q == 11 ? 0.47139673682599764856f
           : q == 12 ? 0.38268343236508977173f
           : q == 13 ? 0.29028467725446236764f
           : q == 14 ? 0.19509032201612826785f
           : q == 15 ? 0.09801714032956060199f
                     : 0.0f;
}
__host__ __device__ constexpr float cos64(int q)
{
    q &= 63;
    if (q > 32) q = 64 - q;
    return q <= 16 ? cos64_table(q) : -cos64_table(32 - q);
}
__host__ __device__ constexpr float sin64(int q)
{
    return cos64(q - 16);
}

template <int R>
__host__ __device__ constexpr int bitrev(int i)
{
    int r = 0;
    for (int b = 1; b < R; b <<= 1) {
        r = (r << 1) | (i & 1);
        i >>= 1;
    }
    return r;
}

// One DIT butterfly with twiddle W = exp(-2*pi*i*q/32) on v:  (u, v) -> (u + v*W, u - v*W).
// General W: u + v*W is two chained FFMA2 (v*(c,c) + (vi,-vr)*(s,s) + u) and the other output
// is 2u - (u + v*W), one more FFMA2: three packed instructions instead of four.
__device__ __forceinline__ void dit_butterfly(c64& u, c64& v, int q)
{
    if (q == 0) {
        const c64 s = cadd(u, v);
        v = csub(u, v);
        u = s;
        return;
    }
    float vr, vi;
    cunpack(v, vr, vi);
    if (q == 8) {                            // v * (-i) = (vi, -vr)
        const c64 t = cpack(vi, -vr);
        const c64 s = cadd(u, t);
        v = csub(u, t);
        u = s;
        return;
    }
    const float c = cos32(q);
    const float sn = sin32(q);
    const c64 s = cfma2(v, cpack(c, c), cfma2(cpack(vi, -vr), cpack(sn, sn), u));
    float sr, si;
    cunpack(s, sr, si);
    v = cfma2(u, cpack(2.0f, 2.0f), cpack(-sr, -si));
    u = s;
}

// First DIT stage with per-input complex pre-multipliers (the inter-pass twiddles):
// (a, b) -> (ta*a + tb*b, ta*a - tb*b) in five packed instructions (three when ta == 1).
__device__ __forceinline__ void dit_butterfly_pretwiddled(c64& a, c64& b, bool a_unit, float2 ta, float2 tb)
{
    c64 p = a;
    if (!a_unit) p = cmul(a, ta.x, ta.y);
    float br, bi;
    cunpack(b, br, bi);
    const c64 s = cfma2(b, cpack(tb.x, tb.x), cfma2(cpack(-bi, br), cpack(tb.y, tb.y), p));
    float sr, si;
    cunpack(s, sr, si);
    b = cfma2(p, cpack(2.0f, 2.0f), cpack(-sr, -si));
    a = s;
}

// In-place forward DIT FFT of 32 points.  Input: a[p] = x[bitrev<32>(p)] (bit-reversed order);
// output in natural order a[k] = X[k].  If PRETW, input x[n] is first multiplied by tw[n]
// (tw[0] is taken as 1), fused into the first stage.
template <bool PRETW>
__device__ __forceinline__ void fft_dit32(c64 (&a)[32], const float2 (&tw)[32])
{
#pragma unroll
    for (int g = 0; g < 32; g += 2) {
        if (PRETW) {
            const int na = bitrev<32>(g);
            const int nb = bitrev<32>(g + 1);
            dit_butterfly_pretwiddled(a[g], a[g + 1], na == 0, tw[na], tw[nb]);
        } else {
            dit_butterfly(a[g], a[g + 1], 0);
        }
    }
#pragma unroll
    for (int half = 2; half <= 16; half <<= 1) {
#pragma unroll
        for (int g = 0; g < 32; g += 2 * half) {
#pragma unroll
            for (int k = 0; k < half; ++k) dit_butterfly(a[g + k], a[g + k + half], k * (16 / half));
        }
    }
}

// The same 32-point transform with the pre-multipliers handed over C floats at a time, in the
// order the first stage consumes them: floats 2g, 2g + 1 of the sequence are re, im of the
// multiplier of input bitrev<32>(g) = register g (g = 0 is taken as 1; its pair is never read), so
// chunk c covers registers C/2 c .. C/2 (c + 1) - 1.  fetch(c, tw) must leave chunk c in tw; it is
// called for c = 0, 1, ... just before the butterflies that need the chunk, so only C registers
// ever hold multipliers instead of the 62 a lane-private copy costs (chain_fused.cu reads them from
// tensor memory).
template <int C, class Fetch>
__device__ __forceinline__ void fft_dit32_pretwiddled_chunks(c64 (&a)[32], uint32_t (&tw)[C], Fetch&& fetch)
{
    static_assert(C % 4 == 0 && 64 % C == 0, "a chunk holds whole butterflies");
#pragma unroll
    for (int c = 0; c < 64 / C; ++c) {
        fetch(c, tw);
#pragma unroll
        for (int j = 0; j < C; j += 4) {
            const int g = (C * c + j) / 2;
            const float2 ta = make_float2(__uint_as_float(tw[j]), __uint_as_float(tw[j + 1]));
            const float2 tb = make_float2(__uint_as_float(tw[j + 2]), __uint_as_float(tw[j + 3]));
            dit_butterfly_pretwiddled(a[g], a[g + 1], g == 0, ta, tb);
        }
    }
#pragma unroll
    for (int half = 2; half <= 16; half <<= 1) {
#pragma unroll
        for (int g = 0; g < 32; g += 2 * half) {
#pragma unroll
            for (int k = 0; k < half; ++k) dit_butterfly(a[g + k], a[g + k + half], k * (16 / half));
        }
    }
}

// DIT butterfly with twiddle exp(-2*pi*i*q/64), 0 <= q < 32 (same three-instruction form)
__device__ __forceinline__ void dit_butterfly64(c64& u, c64& v, int q)
{
    if ((q & 1) == 0) {
        dit_butterfly(u, v, q >> 1);
        return;
    }
    float vr, vi;
    cunpack(v, vr, vi);
    const float c = cos64(q);
    const float sn = sin64(q);
    const c64 s = cfma2(v, cpack(c, c), cfma2(cpack(vi, -vr), cpack(sn, sn), u));
    float sr, si;
    cunpack(s, sr, si);
    v = cfma2(u, cpack(2.0f, 2.0f), cpack(-sr, -si));
    u = s;
}

// In-place forward DIT FFT of 64 points.  Input a[p] = x[bitrev<64>(p)], output natural order.
__device__ __forceinline__ void fft_dit64(c64 (&a)[64])
{
#pragma unroll
    for (int half = 1; half < 64; half <<= 1) {
#pragma unroll
        for (int g = 0; g < 64; g += 2 * half) {
#pragma unroll
            for (int k = 0; k < half; ++k) dit_butterfly64(a[g + k], a[g + k + half], k * (32 / half));
        }
    }
}

// 64-point forward DIT FFT whose input x[n] is first multiplied by tw_col[stride * n] (tw_col[0] taken
// as 1): the inter-pass twiddles of a 64 x 64 decomposition, read just in time from a table column
// (shared memory; consecutive threads read consecutive entries) and fused into the first butterfly
// stage, so they never occupy more than a few registers.
// Input a[p] = x[bitrev<64>(p)], output natural order.
__device__ __forceinline__ void fft_dit64_pretwiddled(c64 (&a)[64], const float2* tw_col, int stride)
{
#pragma unroll
    for (int g = 0; g < 64; g += 2) {
        const int na = bitrev<64>(g);
        const int nb = bitrev<64>(g + 1);
        const float2 ta = na == 0 ? make_float2(1.0f, 0.0f) : tw_col[stride * na];
        const float2 tb = tw_col[stride * nb];
        dit_butterfly_pretwiddled(a[g], a[g + 1], na == 0, ta, tb);
    }
#pragma unroll
    for (int half = 2; half < 64; half <<= 1) {
#pragma unroll
        for (int g = 0; g < 64; g += 2 * half) {
#pragma unroll
            for (int k = 0; k < half; ++k) dit_butterfly64(a[g + k], a[g + k + half], k * (32 / half));
        }
    }
}

// In-place forward DIT FFT of R <= 16 points, no pre-twiddles.  Input a[p] = x[bitrev<R>(p)],
// output natural order.
template <int R>
__device__ __forceinline__ void fft_dit_small(c64 (&a)[R])
{
    static_assert(R == 2 || R == 4 || R == 8 || R == 16, "small register FFT sizes");
#pragma unroll
    for (int half = 1; half < R; half <<= 1) {
#pragma unroll
        for (int g = 0; g < R; g += 2 * half) {
#pragma unroll
            for (int k = 0; k < half; ++k) dit_butterfly(a[g + k], a[g + k + half], k * (16 / half));
        }
    }
}

}  // namespace b200

// fft1024_warp.cuh -- one warp transforms one 1024-point frame held in shared memory
// (shared by spectrum1024.cu and chain_fused.cu).
//
// Decomposition 1024 = 32 x 32 with n = 32*n1 + n2, k = k1 + 32*k2:
//   pass 1: lane n2 holds x[32*n1 + n2] (n1 = 0..31) in registers, 32-point FFT over n1,
//           multiply by W_1024^(n2*k1) (lane-private twiddles kept in registers for the
//           life of the persistent warp), write row k1 of a padded shared tile;
//   pass 2: lane k1 reads its row (all n2), 32-point FFT over n2 -> bins k1 + 32*k2.
// One shared-memory exchange per frame, warp-private (only __syncwarp).
#pragma once

#include "b200_common.cuh"
#include "fft_regs.cuh"

namespace b200 {

constexpr int FFT1024_XCH_STRIDE = 34;                         // float2 per row: LDS.128 / STS.64 conflict-free
constexpr int FFT1024_XCH_BYTES = 32 * FFT1024_XCH_STRIDE * 8;  // 8704 per warp
constexpr float DB_PER_LOG2 = 3.01029995663981195f;            // 10 * log10(2)
// The unpack leaves samples as (x - 128) * 256 (see fft1024_load); the reference wants
// (x - 128) / 128 (spectrum.c:56-57): a factor 2^15 in amplitude, 2^30 in power -- exact.
constexpr float FFT1024_POWER_SCALE = 1.0f / 1073741824.0f;
constexpr float FFT1024_DB_SHIFT = -30.0f * DB_PER_LOG2;       // added to 10*log10(g/K)

// lane-private inter-pass twiddles W_1024^(lane * k1), k1 = 1..31
__device__ __forceinline__ void fft1024_load_twiddles(const float2* __restrict__ table, int lane, float2 (&tw)[32])
{
    tw[0] = make_float2(1.0f, 0.0f);
#pragma unroll
    for (int k1 = 1; k1 < 32; ++k1) tw[k1] = __ldg(&table[(lane * k1) & 1023]);
}

// Unpack (spectrum.c:54-58).  A byte b OR-ed into mantissa bits 8..15 of 2^23 reads as the
// float 2^23 + 256*b, exactly.  All values stay multiples of 256 below 2^29, so the +-
// butterflies of pass 1 are exact on the BIASED values: differences are clean, sums carry the
// bias along the all-sums path only, and just one output (k1 = 0) ends up holding
// 32 * (2^23 + 256*128), which fft1024_core removes with a single subtraction instead of one
// per sample.  With a window the bias has to go before the multiply.
template <bool WINDOW>
__device__ __forceinline__ void fft1024_load(const uint16_t* in16, const float* win, int lane, c64 (&a)[32])
{
    const c64 bias1 = cpack(8421376.0f, 8421376.0f);               // 2^23 + 256 * 128
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) {
        const uint32_t v = in16[32 * n1 + lane];
        const int r = bitrev<32>(n1);          // DIT wants its input in bit-reversed register order
        a[r] = cpack(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7504)),
                     __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7514)));
        if (WINDOW) {
            const float w = win[32 * n1 + lane];
            a[r] = cmul2(csub(a[r], bias1), cpack(w, w));
        }
    }
}

// Both passes.  `a` as left by fft1024_load (or any loader that fills a[bitrev<32>(n1)] with
// sample 32*n1 + lane).  On return b[k2] = X[lane + 32 * k2].  xch: this warp's exchange tile.
// The caller must __syncwarp() between the last read of the frame bytes and anything that
// overwrites them; xch reuse across frames is ordered by the __syncwarp() before the writes.
// The inter-pass twiddles W_1024^(n2*k1) are applied on the READ side (lane = k1, register
// n2 -- the table is symmetric, so the same lane-private tw[] serves) fused into pass 2's first
// butterfly stage.
// first pass: 32-point transforms over n1 (registers only; no twiddles are applied here)
template <bool BIASED>
__device__ __forceinline__ void fft1024_pass1(c64 (&a)[32])
{
    float2 unused[32];
    fft_dit32<false>(a, unused);
    if (BIASED) a[0] = csub(a[0], cpack(269484032.0f, 269484032.0f));   // 32 * (2^23 + 2^15)
}

// transpose through xch + second pass; `a` as left by fft1024_pass1
__device__ __forceinline__ void fft1024_pass2(c64 (&a)[32], const float2 (&tw)[32], float2* xch, int lane, c64 (&b)[32])
{
    __syncwarp();           // every lane is done reading xch for the previous frame
    // stored as float2 halves on purpose: a 64-bit store of the packed register makes ptxas copy every
    // value that was also unpacked (the "2u - s" butterflies) into a scratch pair first -- 38 MOVs per frame
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) {
        float re, im;
        cunpack(a[k1], re, im);
        xch[k1 * FFT1024_XCH_STRIDE + lane] = make_float2(re, im);
    }
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&xch[lane * FFT1024_XCH_STRIDE + 2 * m]);
        b[bitrev<32>(2 * m)] = v.x;
        b[bitrev<32>(2 * m + 1)] = v.y;
    }
    fft_dit32<true>(b, tw);
}

template <bool BIASED>
__device__ __forceinline__ void fft1024_transform(c64 (&a)[32], const float2 (&tw)[32], float2* xch, int lane,
                                                  c64 (&b)[32])
{
    fft1024_pass1<BIASED>(a);
    fft1024_pass2(a, tw, xch, lane, b);
}

// transform + |X|^2:  pw[k2] = |X[lane + 32 * k2]|^2 * 2^30 (raw power)
template <bool BIASED>
__device__ __forceinline__ void fft1024_core(c64 (&a)[32], const float2 (&tw)[32], float2* xch, int lane,
                                             float (&pw)[32])
{
    c64 b[32];
    fft1024_transform<BIASED>(a, tw, xch, lane, b);
#pragma unroll
    for (int k2 = 0; k2 < 32; ++k2) {
        float re, im;
        cunpack(b[k2], re, im);
        pw[k2] = fmaf(re, re, im * im);
    }
}

// display column (fftshift: spectrum.c:25) of pw[k2] for this lane, minus the lane itself
__host__ __device__ constexpr int fft1024_col(int k2)
{
    return 32 * ((k2 + 16) & 31);
}

// Tensor-memory table of the inter-pass twiddles: lane k1 of the warp's quadrant holds, in columns
// 2g and 2g + 1, re and im of W_1024^(k1 * bitrev<32>(g)) for g = 0..31 (g = 0: 1) -- the order
// fft_dit32_pretwiddled_chunks consumes them.  FFT1024_TMEM_COLS columns per lane.
constexpr int FFT1024_TMEM_COLS = 64;
// Columns per tcgen05.ld.  16 and not 32: at 18 warps per SM a thread has 96 registers (five warps share
// one scheduler's 16 K), and 32 twiddle registers next to the 64 of the frame make ptxas spill.
constexpr int FFT1024_TMEM_CHUNK = 16;

// this lane's row of the table, FFT1024_TMEM_CHUNK columns at a time
__device__ __forceinline__ void fft1024_tmem_twiddles(const float2* __restrict__ table, int lane, int c,
                                                      uint32_t (&r)[FFT1024_TMEM_CHUNK])
{
#pragma unroll
    for (int j = 0; j < FFT1024_TMEM_CHUNK; j += 2) {
        const int g = (FFT1024_TMEM_CHUNK * c + j) / 2;
        const float2 w = g == 0 ? make_float2(1.0f, 0.0f) : __ldg(&table[(lane * bitrev<32>(g)) & 1023]);
        r[j] = __float_as_uint(w.x);
        r[j + 1] = __float_as_uint(w.y);
    }
}

// pass 2 with the inter-pass twiddles in tensor memory; tw_taddr = column 0 of this warp's quadrant of the
// table.  The first chunk is requested before the exchange, so its latency hides behind the exchange's loads;
// the other three are requested one at a time, each just before its four butterflies (tcgen05.wait::ld waits
// for every outstanding load, and a second chunk in flight would not fit in the registers either).
__device__ __forceinline__ void fft1024_pass2_tmem_tw(c64 (&a)[32], uint32_t tw_taddr, float2* xch, int lane,
                                                      c64 (&b)[32])
{
    uint32_t tw[FFT1024_TMEM_CHUNK];
    tmem_ld_32x32b_x16(tw_taddr, tw);
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) {
        float re, im;
        cunpack(a[k1], re, im);
        xch[k1 * FFT1024_XCH_STRIDE + lane] = make_float2(re, im);
    }
    __syncwarp();
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&xch[lane * FFT1024_XCH_STRIDE + 2 * m]);
        b[bitrev<32>(2 * m)] = v.x;
        b[bitrev<32>(2 * m + 1)] = v.y;
    }
    fft_dit32_pretwiddled_chunks(b, tw, [&](int c, uint32_t (&r)[FFT1024_TMEM_CHUNK]) {
        if (c > 0) tmem_ld_32x32b_x16(tw_taddr + FFT1024_TMEM_CHUNK * c, r);
        tmem_wait_ld(r);
    });
}

// |X|^2 of the transform's output, as raw power (see FFT1024_POWER_SCALE)
__device__ __forceinline__ void fft1024_power(const c64 (&b)[32], float (&pw)[32])
{
#pragma unroll
    for (int k2 = 0; k2 < 32; ++k2) {
        float re, im;
        cunpack(b[k2], re, im);
        pw[k2] = fmaf(re, re, im * im);
    }
}

// dB rows (cbb_main.c:125 without the truncation): 10*log10(pw) + dboff for two bins per packed FMA
__device__ __forceinline__ void fft1024_store_db(float* out_lane, const float (&pw)[32], float dboff)
{
    const c64 scale = cpack(DB_PER_LOG2, DB_PER_LOG2);
    const c64 off = cpack(dboff, dboff);
#pragma unroll
    for (int k2 = 0; k2 < 32; k2 += 2) {
        float d0, d1;
        cunpack(cfma2(cpack(lg2_ftz(pw[k2]), lg2_ftz(pw[k2 + 1])), scale, off), d0, d1);
        __stcs(out_lane + fft1024_col(k2), d0);
        __stcs(out_lane + fft1024_col(k2 + 1), d1);
    }
}

}  // namespace b200

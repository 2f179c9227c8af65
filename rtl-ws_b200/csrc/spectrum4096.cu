// spectrum4096.cu -- batched 4096-point power spectra (BASELINE config 2's second size), two warps
// per frame, 64 points per thread (sm_100a).
//
// 4096 = 64 x 64 with n = 64*n1 + n2, k = k1 + 64*k2:
//   pass 1: thread n2 (0..63) holds x[64*n1 + n2] (n1 = 0..63) in registers and runs a 64-point
//           FFT over n1 (fft_dit64: 128 registers of data);
//   one exchange through a shared tile (unpadded, XOR-swizzled: the 64-bit column stores and the
//           128-bit row loads are both conflict-free);
//   pass 2: thread k1 reads its row, multiplies by W_4096^(n2*k1) -- a [n2][k1] table the CTA
//           keeps in shared memory, fused into the first butterfly stage -- and runs a 64-point
//           FFT over n2: bins k1 + 64*k2, so a warp store is 128 contiguous bytes.
// Against running four 1024-point branch transforms and a radix-4 combine (spectrum_mx1024.cu)
// this needs ONE shared-memory round trip per point instead of two (the exchange traffic is what
// saturates first there: 346 shared wavefronts per 1024 points against 232 here) and about 30 %
// fewer instructions per sample.
//
// One CTA per SM holds FOUR independent frame pairs (own ring, own tile, own barriers) that share
// the 32 KB twiddle table: with the table in global memory (two-warp CTAs) ncu showed it missing
// L1 -- 28 KB is all that is left next to 200 KB of shared memory -- and the second pass starting
// on L2 latency (585 Gsamples/s; 675 with the table in shared memory).
// The two warps of a frame meet twice per frame on mbarriers: `tfull` once both have stored their
// pass-1 columns, and `tdone` -- on which they arrive as soon as their rows are in registers and
// wait only before the NEXT frame's column stores, a whole second pass, epilogue, gather and first
// pass later.  Frames arrive by TMA bulk copies into a two-deep ring per pair.
//
// Reference arithmetic per frame as in spectrum1024.cu: spectrum.c:54-58 (unpack), :21 (forward
// DFT), :23-34 (fftshift, |X|^2, accumulate, DC-position patch), cbb_main.c:112-128 (dB, u8).
// The DC position (display index N/2) repeats bin N-1, which thread 63 owns: it stores that
// value twice, thread 0 skips its own bin 0 -- no hand-over between threads.
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

constexpr int N4K = 4096;
constexpr int S4K_PAIRS = 4;                                         // frame pairs (2 warps each) per CTA
constexpr int S4K_THREADS = 64 * S4K_PAIRS;
constexpr int S4K_FRAME_BYTES = 2 * N4K;
constexpr int S4K_STAGES = 2;
constexpr int S4K_TILE_BYTES = 64 * 64 * 8;                          // 32768: unpadded, XOR-swizzled (see tile_col)
constexpr int S4K_TW_BYTES = 64 * 64 * 8;                            // the [n2][k1] inter-pass twiddle table
constexpr int S4K_PAIR_BYTES = S4K_STAGES * S4K_FRAME_BYTES + S4K_TILE_BYTES;
constexpr int S4K_BAR_OFFSET = S4K_TW_BYTES + S4K_PAIRS * S4K_PAIR_BYTES;
constexpr int S4K_BAR_BYTES = 64;                                    // per pair: full[2], tfull, tdone
constexpr int S4K_SMEM = S4K_BAR_OFFSET + S4K_PAIRS * S4K_BAR_BYTES;  // 229632 of the 232448 a CTA may have

// Exchange-tile column of element (row, col): columns are XOR-ed with 2 * (row mod 8).  A column store
// (fixed row, 32 consecutive cols) stays a permutation of 32 consecutive 8-byte slots; a 128-bit row
// load (32 consecutive rows, the pair 2m, 2m+1) lands its 8 lanes per quarter-warp on 8 different
// 16-byte slots.  Both conflict-free without padding, which is what lets four tiles, four two-deep
// rings and the twiddle table share one SM.
__device__ __forceinline__ int tile_col(int row, int col)
{
    return col ^ (2 * (row & 7));
}

// pw[k2] = raw power of bin t + 64*k2 -> the requested arrays, display order: col = t + 64*((k2 + 32) & 63).
// `base` = row * 4096 + t.  dc: the value for display index 2048 (written by thread 63 only).
__device__ __forceinline__ void store_row4096(const SpecParams& p, float dboff, size_t base, int t, const float (&pw)[64],
                                              float dc)
{
    if (p.db != nullptr) {
        float* out = p.db + base;
#pragma unroll
        for (int k2 = 0; k2 < 64; ++k2) {
            const float v = fmaf(DB_PER_LOG2, lg2_ftz(pw[k2]), dboff);
            if (k2 != 0 || t != 0) __stcs(out + 64 * ((k2 + 32) & 63), v);
        }
        if (t == 63) __stcs(out + (2048 - 63), fmaf(DB_PER_LOG2, lg2_ftz(dc), dboff));
    }
    if (p.power != nullptr) {
        float* out = p.power + base;
#pragma unroll
        for (int k2 = 0; k2 < 64; ++k2)
            if (k2 != 0 || t != 0) __stcs(out + 64 * ((k2 + 32) & 63), pw[k2] * FFT1024_POWER_SCALE);
        if (t == 63) __stcs(out + (2048 - 63), dc * FFT1024_POWER_SCALE);
    }
    if (p.db_u8 != nullptr) {
        uint8_t* out = p.db_u8 + base;
        // cbb_main.c:125-127: (int) truncation toward zero, then clamp; -inf / NaN -> 0
        auto u8 = [&](float x) {
            int m = __float2int_rz(fmaf(DB_PER_LOG2, lg2_ftz(x), dboff));
            m = m < 0 ? 0 : (m > 255 ? 255 : m);
            return (uint8_t) m;
        };
#pragma unroll
        for (int k2 = 0; k2 < 64; ++k2)
            if (k2 != 0 || t != 0) out[64 * ((k2 + 32) & 63)] = u8(pw[k2]);
        if (t == 63) out[2048 - 63] = u8(dc);
    }
}

template <bool WINDOW, bool MULTI>
__global__ void __launch_bounds__(S4K_THREADS, 1) spectrum4096_kernel(const SpecParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int pair = threadIdx.x >> 6;
    const int t = threadIdx.x & 63;
    const int lane = t & 31;
    float2* tws = reinterpret_cast<float2*>(smem);                                  // [n2][k1]
    uint8_t* ring = smem + S4K_TW_BYTES + pair * S4K_PAIR_BYTES;
    c64* tile = reinterpret_cast<c64*>(ring + S4K_STAGES * S4K_FRAME_BYTES);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + S4K_BAR_OFFSET + pair * S4K_BAR_BYTES);
    uint64_t* tfull = full + S4K_STAGES;
    uint64_t* tdone = tfull + 1;

    const uint32_t total_items = (uint32_t) p.n_streams * (uint32_t) p.n_rows;
    const uint32_t n_rows = (uint32_t) p.n_rows;
    const int K = MULTI ? p.K : 1;
    const uint32_t first = blockIdx.x * S4K_PAIRS + pair;              // pairs stride over rows like CTAs would
    const uint32_t stride = gridDim.x * S4K_PAIRS;
    const uint32_t n_items = first < total_items ? (total_items - first + stride - 1) / stride : 0;
    const uint32_t n_frames = n_items * (uint32_t) K;

    for (int i = threadIdx.x; i < 64 * 64; i += S4K_THREADS) tws[i] = __ldg(p.twiddle_n + i);
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < S4K_STAGES; ++i) mbar_init(&full[i], 1);
        mbar_init(tfull, 2);
        mbar_init(tdone, 2);
        fence_mbar_init();
    }
    __syncthreads();

    auto frame_src = [&](uint32_t f) -> const uint8_t* {
        const uint32_t item = first + (f / (uint32_t) K) * stride;
        const uint32_t j = f % (uint32_t) K;
        const uint32_t s = item / n_rows;
        const uint32_t row = item - s * n_rows;
        return p.iq + (int64_t) s * p.stream_stride_bytes + 2 * ((int64_t) row * p.row_hop + (int64_t) j * p.hop);
    };
    if (t == 0) {
        for (uint32_t f = 0; f < (uint32_t) S4K_STAGES && f < n_frames; ++f) {
            mbar_arrive_expect_tx(&full[f], S4K_FRAME_BYTES);
            tma_load_1d(ring + f * S4K_FRAME_BYTES, frame_src(f), S4K_FRAME_BYTES, &full[f]);
        }
    }

    const float2* twcol = tws + t;                            // W_4096^(n2 * t) at [n2][t]
    // The periodic Hann window of sample 64*n1 + t, without a table:  w = 1/2 - 1/2 cos(2 pi (64 n1 + t) / 4096)
    //   = 1/2 - 1/2 (cos(2 pi n1 / 64) * ct - sin(2 pi n1 / 64) * st),  ct, st = cos, sin(2 pi t / 4096):
    // two FMAs with compile-time coefficients per sample (a 16 KB table next to 224 KB of shared memory would
    // come from L2 every time: 521 Gsamples/s with the table, measured).
    float ct = 1.0f, st = 0.0f;
    if (WINDOW) sincospif((float) t * (1.0f / 2048.0f), &st, &ct);
    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;

    float acc[64];          // MULTI only (dead otherwise)
    if (MULTI) {
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] = 0.0f;
    }
    float dcacc = 0.0f;

    uint32_t f = 0;
    for (uint32_t it = 0; it < n_items; ++it) {
        const uint32_t item = first + it * stride;
        const size_t out_base = (size_t) item * N4K + (size_t) t;
        for (int j = 0; j < K; ++j, ++f) {
            const int stage = f % S4K_STAGES;
            mbar_wait(&full[stage], (f / S4K_STAGES) & 1);
            const uint16_t* in16 = reinterpret_cast<const uint16_t*>(ring + stage * S4K_FRAME_BYTES);

            // ---- pass 1: column t, samples 64*n1 + t ----
            c64 a[64];
            {
                const c64 bias1 = cpack(8421376.0f, 8421376.0f);           // 2^23 + 256 * 128
#pragma unroll
                for (int n1 = 0; n1 < 64; ++n1) {
                    const uint32_t v = in16[64 * n1 + t];
                    const int q = bitrev<64>(n1);
                    a[q] = cpack(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7504)),
                                 __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7514)));
                    if (WINDOW) {
                        const float w = fmaf(0.5f * sin64(n1), st, fmaf(-0.5f * cos64(n1), ct, 0.5f));
                        a[q] = cmul2(csub(a[q], bias1), cpack(w, w));
                    }
                }
            }
            fft_dit64(a);
            // the biased unpack (fft1024_load) leaves 64 * (2^23 + 2^15) on the all-sums output only
            if (!WINDOW) a[0] = csub(a[0], cpack(538968064.0f, 538968064.0f));

            if (f > 0) mbar_wait(tdone, (f - 1) & 1);         // both warps hold their rows of frame f - 1
#pragma unroll
            for (int k1 = 0; k1 < 64; ++k1) cstore(&tile[k1 * 64 + tile_col(k1, t)], a[k1]);
            __syncwarp();
            if (lane == 0) mbar_arrive(tfull);
            mbar_wait(tfull, f & 1);
            if (t == 0 && f + S4K_STAGES < n_frames) {        // both warps have consumed the stage
                fence_proxy_async_smem();
                mbar_arrive_expect_tx(&full[stage], S4K_FRAME_BYTES);
                tma_load_1d(ring + stage * S4K_FRAME_BYTES, frame_src(f + S4K_STAGES), S4K_FRAME_BYTES, &full[stage]);
            }

            // ---- pass 2: row t ----
            c64 b[64];
#pragma unroll
            for (int m = 0; m < 32; ++m) {
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&tile[t * 64 + tile_col(t, 2 * m)]);
                b[bitrev<64>(2 * m)] = v.x;
                b[bitrev<64>(2 * m + 1)] = v.y;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(tdone);
            fft_dit64_pretwiddled(b, twcol, 64);

            float pw[64];
#pragma unroll
            for (int k2 = 0; k2 < 64; ++k2) {
                float re, im;
                cunpack(b[k2], re, im);
                pw[k2] = fmaf(re, re, im * im);
            }
            if (!MULTI) {
                store_row4096(p, dboff, out_base, t, pw, pw[63]);
            } else {
#pragma unroll
                for (int k2 = 0; k2 < 64; ++k2) acc[k2] += pw[k2];
                dcacc = fmaf((float) (K - j), pw[63], dcacc);   // thread 63: sum_j (K - j) |X_j[N-1]|^2
            }
        }
        if (MULTI) {
            store_row4096(p, dboff, out_base, t, acc, dcacc);
#pragma unroll
            for (int k2 = 0; k2 < 64; ++k2) acc[k2] = 0.0f;
            dcacc = 0.0f;
        }
    }
}

}  // namespace

// N = 4096, cmplx_u8 input.  p.twiddle_n must be the [64][64] table W_4096^(n2 * k1).  A non-null p.window
// means the periodic Hann window (the only one b200_spectrum_plan_create offers); the kernel computes it.
int launch_spectrum4096(const SpecParams& p, cudaStream_t stream)
{
    const uint64_t total = (uint64_t) p.n_streams * (uint64_t) p.n_rows;
    auto kern = p.K > 1 ? (p.window ? spectrum4096_kernel<true, true> : spectrum4096_kernel<false, true>)
                        : (p.window ? spectrum4096_kernel<true, false> : spectrum4096_kernel<false, false>);
    if (int rc = ensure_dynamic_smem((const void*) kern, S4K_SMEM)) return rc;
    uint64_t grid = (uint64_t) sm_count();                     // one CTA of four frame pairs per SM
    const uint64_t needed = (total + S4K_PAIRS - 1) / S4K_PAIRS;
    if (grid > needed) grid = needed;
    kern<<<(unsigned) grid, S4K_THREADS, S4K_SMEM, stream>>>(p);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

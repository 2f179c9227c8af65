// spectrum2048.cu -- batched 2048-point power spectra, one warp per frame, no inter-warp synchronisation
// (sm_100a).
//
// 2048 = 64 x 32 with n = 32*n1 + n2, k = k1 + 64*k2:
//   pass 1: lane n2 holds x[32*n1 + n2] (n1 = 0..63) in registers and runs a 64-point FFT over n1
//           (fft_dit64: 128 registers of data);
//   one warp-private exchange through a shared tile of 64 rows x 32 columns (unpadded, XOR-swizzled);
//   pass 2: lane l takes the two rows k1 = l and k1 = l + 32 one after the other: multiply by
//           W_2048^(n2*k1) -- a [n2][k1] table the CTA keeps in shared memory, fused into the first
//           butterfly stage -- and a 32-point FFT over n2: bins k1 + 64*k2.  For a fixed k2 the warp
//           stores 32 consecutive bins, twice.
// Same idea as spectrum4096.cu (64 points per thread, one shared-memory round trip per point instead of the
// two of the M-branch kernel), but a frame fits one warp here, so there is nothing to wait for except the
// TMA copy of the next frame (two-deep warp-private ring).  Eight warps per SM at <= 255 registers.
//
// Reference arithmetic per frame as in spectrum1024.cu: spectrum.c:54-58 (unpack), :21 (forward DFT), :23-34
// (fftshift, |X|^2, accumulate, DC-position patch), cbb_main.c:112-128 (dB, u8).
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

constexpr int N2K = 2048;
constexpr int S2K_WARPS = 8;
constexpr int S2K_THREADS = S2K_WARPS * 32;
constexpr int S2K_FRAME_BYTES = 2 * N2K;                             // 4096
constexpr int S2K_TILE_BYTES = 64 * 32 * 8;                          // 16384
constexpr int S2K_TW_BYTES = 32 * 64 * 8;                            // [n2][k1] inter-pass twiddles
constexpr int S2K_WARP_BYTES = 2 * S2K_FRAME_BYTES + S2K_TILE_BYTES + 32;   // ring, tile, 2 mbarriers (+pad)
constexpr int S2K_SMEM = S2K_TW_BYTES + S2K_WARPS * S2K_WARP_BYTES;

// Tile element (row k1, column n2) lives in column n2 ^ (2 * (k1 & 7)) -- see spectrum4096.cu: column stores of
// one row stay a permutation of 32 consecutive slots, 128-bit row loads of 8 consecutive rows hit 8 different
// 16-byte slots.
__device__ __forceinline__ int tile_col2k(int row, int col)
{
    return col ^ (2 * (row & 7));
}

// 32-point DIT FFT with the inter-pass twiddles read from a table column in shared memory (stride in entries)
__device__ __forceinline__ void fft_dit32_pretwiddled_smem(c64 (&a)[32], const float2* tw_col, int stride)
{
#pragma unroll
    for (int g = 0; g < 32; g += 2) {
        const int na = bitrev<32>(g);
        const int nb = bitrev<32>(g + 1);
        const float2 ta = na == 0 ? make_float2(1.0f, 0.0f) : tw_col[stride * na];
        const float2 tb = tw_col[stride * nb];
        dit_butterfly_pretwiddled(a[g], a[g + 1], na == 0, ta, tb);
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

// pw[k2] = raw power of bin k1 + 64*k2 for this lane's row k1 = lane + 32*h -> display order:
// col = (k + 1024) & 2047 = k1 + 64 * ((k2 + 16) & 31).  `base` = row * 2048 + k1.
// skip0: this lane owns bin 0 (k1 = 0, k2 = 0), whose display slot takes bin N-1's value instead.
__device__ __forceinline__ void store_half2048(const SpecParams& p, float dboff, size_t base, const float (&pw)[32], bool skip0)
{
    if (p.db != nullptr) {
        float* out = p.db + base;
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2)
            if (k2 != 0 || !skip0) __stcs(out + 64 * ((k2 + 16) & 31), fmaf(DB_PER_LOG2, lg2_ftz(pw[k2]), dboff));
    }
    if (p.power != nullptr) {
        float* out = p.power + base;
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2)
            if (k2 != 0 || !skip0) __stcs(out + 64 * ((k2 + 16) & 31), pw[k2] * FFT1024_POWER_SCALE);
    }
    if (p.db_u8 != nullptr) {
        uint8_t* out = p.db_u8 + base;
#pragma unroll
        for (int k2 = 0; k2 < 32; ++k2) {
            // cbb_main.c:125-127: (int) truncation toward zero, then clamp; -inf / NaN -> 0
            int m = __float2int_rz(fmaf(DB_PER_LOG2, lg2_ftz(pw[k2]), dboff));
            m = m < 0 ? 0 : (m > 255 ? 255 : m);
            if (k2 != 0 || !skip0) out[64 * ((k2 + 16) & 31)] = (uint8_t) m;
        }
    }
}

// the DC position (display index N/2) repeats bin N-1 (spectrum.c:30-33): written by the lane that owns it
__device__ __forceinline__ void store_dc2048(const SpecParams& p, float dboff, size_t row_base, float v)
{
    const float db = fmaf(DB_PER_LOG2, lg2_ftz(v), dboff);
    if (p.db != nullptr) __stcs(p.db + row_base + N2K / 2, db);
    if (p.power != nullptr) __stcs(p.power + row_base + N2K / 2, v * FFT1024_POWER_SCALE);
    if (p.db_u8 != nullptr) {
        int m = __float2int_rz(db);
        m = m < 0 ? 0 : (m > 255 ? 255 : m);
        p.db_u8[row_base + N2K / 2] = (uint8_t) m;
    }
}

template <bool WINDOW, bool MULTI>
__global__ void __launch_bounds__(S2K_THREADS, 1) spectrum2048_kernel(const SpecParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    float2* tws = reinterpret_cast<float2*>(smem);                                  // [n2][k1], 32 x 64
    uint8_t* wbase = smem + S2K_TW_BYTES + warp * S2K_WARP_BYTES;
    uint8_t* ring = wbase;
    c64* tile = reinterpret_cast<c64*>(wbase + 2 * S2K_FRAME_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(wbase + 2 * S2K_FRAME_BYTES + S2K_TILE_BYTES);

    const uint32_t total_items = (uint32_t) p.n_streams * (uint32_t) p.n_rows;
    const uint32_t n_rows = (uint32_t) p.n_rows;
    const int K = MULTI ? p.K : 1;
    const uint32_t gw = blockIdx.x * S2K_WARPS + warp;
    const uint32_t GW = gridDim.x * S2K_WARPS;
    const uint32_t n_items = gw < total_items ? (total_items - gw + GW - 1) / GW : 0;
    const uint32_t n_frames = n_items * (uint32_t) K;

    for (int i = threadIdx.x; i < 32 * 64; i += S2K_THREADS) tws[i] = __ldg(p.twiddle_n + i);
    if (lane == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto frame_src = [&](uint32_t f) -> const uint8_t* {
        const uint32_t item = gw + (f / (uint32_t) K) * GW;
        const uint32_t j = f % (uint32_t) K;
        const uint32_t s = item / n_rows;
        const uint32_t row = item - s * n_rows;
        return p.iq + (int64_t) s * p.stream_stride_bytes + 2 * ((int64_t) row * p.row_hop + (int64_t) j * p.hop);
    };
    if (lane == 0) {
        for (uint32_t f = 0; f < 2 && f < n_frames; ++f) {
            mbar_arrive_expect_tx(&bars[f], S2K_FRAME_BYTES);
            tma_load_1d(ring + f * S2K_FRAME_BYTES, frame_src(f), S2K_FRAME_BYTES, &bars[f]);
        }
    }

    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;
    // periodic Hann of sample 32*n1 + lane, computed: 1/2 - 1/2 (cos(2 pi n1 / 64) ct - sin(2 pi n1 / 64) st)
    float ct = 1.0f, st = 0.0f;
    if (WINDOW) sincospif((float) lane * (1.0f / 1024.0f), &st, &ct);

    float acc[64];          // MULTI only: [h][k2]
    if (MULTI) {
#pragma unroll
        for (int i = 0; i < 64; ++i) acc[i] = 0.0f;
    }
    float dcacc = 0.0f;

    uint32_t f = 0;
    for (uint32_t it = 0; it < n_items; ++it) {
        const uint32_t item = gw + it * GW;
        const size_t row_base = (size_t) item * N2K;
        for (int j = 0; j < K; ++j, ++f) {
            const int stage = f & 1;
            mbar_wait(&bars[stage], (f >> 1) & 1);
            const uint16_t* in16 = reinterpret_cast<const uint16_t*>(ring + stage * S2K_FRAME_BYTES);

            // ---- pass 1: column `lane`, samples 32*n1 + lane ----
            c64 a[64];
            {
                const c64 bias1 = cpack(8421376.0f, 8421376.0f);           // 2^23 + 256 * 128
#pragma unroll
                for (int n1 = 0; n1 < 64; ++n1) {
                    const uint32_t v = in16[32 * n1 + lane];
                    const int q = bitrev<64>(n1);
                    a[q] = cpack(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7504)),
                                 __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7514)));
                    if (WINDOW) {
                        const float w = fmaf(0.5f * sin64(n1), st, fmaf(-0.5f * cos64(n1), ct, 0.5f));
                        a[q] = cmul2(csub(a[q], bias1), cpack(w, w));
                    }
                }
            }
            __syncwarp();
            if (lane == 0 && f + 2 < n_frames) {              // the stage is consumed: request the frame two ahead
                fence_proxy_async_smem();
                mbar_arrive_expect_tx(&bars[stage], S2K_FRAME_BYTES);
                tma_load_1d(ring + stage * S2K_FRAME_BYTES, frame_src(f + 2), S2K_FRAME_BYTES, &bars[stage]);
            }
            fft_dit64(a);
            // the biased unpack leaves 64 * (2^23 + 2^15) on the all-sums output only
            if (!WINDOW) a[0] = csub(a[0], cpack(538968064.0f, 538968064.0f));

            __syncwarp();                                     // every lane has read its rows of the previous frame
#pragma unroll
            for (int k1 = 0; k1 < 64; ++k1) cstore(&tile[k1 * 32 + tile_col2k(k1, lane)], a[k1]);
            __syncwarp();

            // ---- pass 2: rows k1 = lane and lane + 32 ----
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k1 = lane + 32 * h;
                c64 b[32];
#pragma unroll
                for (int m = 0; m < 16; ++m) {
                    const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&tile[k1 * 32 + tile_col2k(k1, 2 * m)]);
                    b[bitrev<32>(2 * m)] = v.x;
                    b[bitrev<32>(2 * m + 1)] = v.y;
                }
                fft_dit32_pretwiddled_smem(b, tws + k1, 64);
                float pw[32];
#pragma unroll
                for (int k2 = 0; k2 < 32; ++k2) {
                    float re, im;
                    cunpack(b[k2], re, im);
                    pw[k2] = fmaf(re, re, im * im);
                }
                // bin N-1 = (k1 63, k2 31): lane 31 in the second half
                if (!MULTI) {
                    store_half2048(p, dboff, row_base + k1, pw, k1 == 0);
                    if (h == 1 && lane == 31) store_dc2048(p, dboff, row_base, pw[31]);
                } else {
#pragma unroll
                    for (int k2 = 0; k2 < 32; ++k2) acc[32 * h + k2] += pw[k2];
                    if (h == 1) dcacc = fmaf((float) (K - j), pw[31], dcacc);       // lane 31: sum_j (K - j) |X_j[N-1]|^2
                }
            }
        }
        if (MULTI) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float pw[32];
#pragma unroll
                for (int k2 = 0; k2 < 32; ++k2) {
                    pw[k2] = acc[32 * h + k2];
                    acc[32 * h + k2] = 0.0f;
                }
                store_half2048(p, dboff, row_base + lane + 32 * h, pw, lane + 32 * h == 0);
            }
            if (lane == 31) store_dc2048(p, dboff, row_base, dcacc);
            dcacc = 0.0f;
        }
    }
}

}  // namespace

// N = 2048, cmplx_u8 input.  p.twiddle_n must be the [32][64] table W_2048^(n2 * k1).  A non-null p.window means
// the periodic Hann window (the only one b200_spectrum_plan_create offers); the kernel computes it.
int launch_spectrum2048(const SpecParams& p, cudaStream_t stream)
{
    const uint64_t total = (uint64_t) p.n_streams * (uint64_t) p.n_rows;
    auto kern = p.K > 1 ? (p.window ? spectrum2048_kernel<true, true> : spectrum2048_kernel<false, true>)
                        : (p.window ? spectrum2048_kernel<true, false> : spectrum2048_kernel<false, false>);
    if (int rc = ensure_dynamic_smem((const void*) kern, S2K_SMEM)) return rc;
    uint64_t grid = (uint64_t) sm_count();                     // one CTA of eight frame-warps per SM
    const uint64_t needed = (total + S2K_WARPS - 1) / S2K_WARPS;
    if (grid > needed) grid = needed;
    kern<<<(unsigned) grid, S2K_THREADS, S2K_SMEM, stream>>>(p);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

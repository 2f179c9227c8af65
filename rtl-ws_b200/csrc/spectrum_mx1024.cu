// spectrum_mx1024.cu -- batched power spectra for N = 8192 = M * 1024, M = 8 (sm_100a): the
// largest frame that still fits one CTA's shared memory.  2048 and 4096 (BASELINE config 2's second
// size) have their own kernels with a single shared-memory round trip (spectrum2048.cu,
// spectrum4096.cu), which measured faster than this form at M = 2 and 4 (637 vs 517 and 675 vs 490
// Gsamples/s).
//
// Decimation in time by M:  X[k + 1024 q] = sum_{r<M} W_M^(r q) * ( W_N^(r k) * F_r[k] ),
// F_r = the 1024-point transform of the polyphase branch x[M m + r].  A CTA is M warps:
//   1. the frame (2N bytes) arrives by one TMA bulk copy (two-deep ring);
//   2. warp r runs the 32x32 register transform of fft1024_warp.cuh on branch r (stride-M u16
//      reads from shared memory), multiplies by W_N^(r k) and parks Z_r[k] in its own exchange
//      tile (the tile is free again after the transform's transpose);
//   3. the warps meet on an mbarrier (the only rendezvous of a frame; exchange tiles alternate
//      between two sets so nothing else needs ordering); every warp takes 1024/M values of k,
//      reads Z_0..Z_{M-1}[k], runs the M-point butterfly in registers and gets bins k, k + 1024,
//      ... : |X|^2, K-frame accumulation with the cumulative DC-position patch
//      (spectrum.c:30-33), dB / power / u8.
// Arithmetic per frame as in spectrum1024.cu (spectrum.c:15-58, cbb_main.c:112-128).
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

constexpr int M = 8;                                 // polyphase branches = warps per CTA
constexpr int N = M * 1024;
constexpr int MX_FRAME_BYTES = 2 * N;
constexpr int MX_THREADS = M * 32;
constexpr int MX_KPW = 32 / M;                       // k-groups of 32 per warp in the combine
constexpr int MX_STAGES = 2;                         // TMA ring
constexpr int MX_TILE_SETS = 2;                      // exchange tiles alternate between frames
constexpr int MX_BAR_OFFSET = MX_STAGES * MX_FRAME_BYTES + MX_TILE_SETS * M * FFT1024_XCH_BYTES;
constexpr int MX_SMEM = MX_BAR_OFFSET + 64;

// 32 output values of one warp (index g * M + q: bin = (r * MX_KPW + g) * 32 + lane + 1024 q) -> the
// requested arrays in display order (fftshift of spectrum.c:25: bin + N/2 mod N moves the q digit
// by M/2).  `base` = row * N + r * MX_KPW * 32 + lane: every store is base + a compile-time offset
// and a warp store covers 128 contiguous bytes.
__device__ __forceinline__ void store_bins(const SpecParams& p, float dboff, size_t base, const float (&pw)[32])
{
    if (p.db != nullptr) {
        float* out = p.db + base;
#pragma unroll
        for (int g = 0; g < MX_KPW; ++g)
#pragma unroll
            for (int q = 0; q < M; ++q)
                __stcs(out + 32 * g + 1024 * ((q + M / 2) % M), fmaf(DB_PER_LOG2, lg2_ftz(pw[g * M + q]), dboff));
    }
    if (p.power != nullptr) {
        float* out = p.power + base;
#pragma unroll
        for (int g = 0; g < MX_KPW; ++g)
#pragma unroll
            for (int q = 0; q < M; ++q) __stcs(out + 32 * g + 1024 * ((q + M / 2) % M), pw[g * M + q] * FFT1024_POWER_SCALE);
    }
    if (p.db_u8 != nullptr) {
        uint8_t* out = p.db_u8 + base;
#pragma unroll
        for (int g = 0; g < MX_KPW; ++g)
#pragma unroll
            for (int q = 0; q < M; ++q) {
                // cbb_main.c:125-127: (int) truncation toward zero, then clamp; -inf / NaN -> 0
                int m = __float2int_rz(fmaf(DB_PER_LOG2, lg2_ftz(pw[g * M + q]), dboff));
                m = m < 0 ? 0 : (m > 255 ? 255 : m);
                out[32 * g + 1024 * ((q + M / 2) % M)] = (uint8_t) m;
            }
    }
}

// Synchronisation: ONE rendezvous per frame and no block barrier.  Frame f uses exchange-tile set
// f & 1 (both for the transform's transpose and for the parked Z_r), and every warp arrives on
// zfull[f & 1] once its Z_r is parked.  A warp that has passed the wait on zfull(f) knows that all
// warps (i) have finished reading frame f's bytes, so thread 0 may hand the stage back to the TMA
// unit, and (ii) had finished combining frame f - 1 before they started on f, so tile set
// (f + 1) & 1 is free to be overwritten: nothing else needs ordering.  Between its arrival and the
// wait a warp gathers the next frame and runs its first pass (registers only).
// One CTA of 8 warps per SM: room for 255 registers per thread.
template <bool WINDOW, bool MULTI>
__global__ void __launch_bounds__(MX_THREADS, 1) spectrum_mx1024_kernel(const SpecParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int r = tid >> 5;                                   // polyphase branch of this warp
    uint8_t* ring = smem;
    uint8_t* tiles = smem + MX_STAGES * MX_FRAME_BYTES;       // [set][branch] tiles of FFT1024_XCH_BYTES
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + MX_BAR_OFFSET);
    uint64_t* zfull = full + MX_STAGES;

    const uint32_t total_items = (uint32_t) p.n_streams * (uint32_t) p.n_rows;
    const uint32_t n_rows = (uint32_t) p.n_rows;
    const int K = MULTI ? p.K : 1;
    if (blockIdx.x >= total_items) return;
    const uint32_t n_items = (total_items - blockIdx.x + gridDim.x - 1) / gridDim.x;
    const uint32_t n_frames = n_items * (uint32_t) K;

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < MX_STAGES; ++i) mbar_init(&full[i], 1);
        mbar_init(&zfull[0], M);
        mbar_init(&zfull[1], M);
        fence_mbar_init();
    }
    __syncthreads();

    auto frame_src = [&](uint32_t f) -> const uint8_t* {
        const uint32_t item = blockIdx.x + (f / (uint32_t) K) * gridDim.x;
        const uint32_t j = f % (uint32_t) K;
        const uint32_t s = item / n_rows;
        const uint32_t row = item - s * n_rows;
        return p.iq + (int64_t) s * p.stream_stride_bytes + 2 * ((int64_t) row * p.row_hop + (int64_t) j * p.hop);
    };
    if (tid == 0) {
        for (uint32_t f = 0; f < (uint32_t) MX_STAGES && f < n_frames; ++f) {
            mbar_arrive_expect_tx(&full[f], MX_FRAME_BYTES);
            tma_load_1d(ring + f * MX_FRAME_BYTES, frame_src(f), MX_FRAME_BYTES, &full[f]);
        }
    }

    float2 tw[32];
    fft1024_load_twiddles(p.twiddle, lane, tw);               // W_1024^(lane * k1)
    const float2* twr = p.twiddle_n + r * 1024 + lane;        // W_N^(r * k), k = lane + 32 * k2
    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;

    float acc[32];
    if (MULTI) {
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
    }
    float dcacc = 0.0f;

    // branch r of a frame: samples M*(32*n1 + lane) + r, then the first pass (32-point transforms
    // over n1, registers only)
    c64 a[32];
    auto gather_pass1 = [&](uint32_t ff) {
        const int st = ff % MX_STAGES;
        mbar_wait(&full[st], (ff / MX_STAGES) & 1);
        const uint16_t* in16 = reinterpret_cast<const uint16_t*>(ring + st * MX_FRAME_BYTES);
        const c64 bias1 = cpack(8421376.0f, 8421376.0f);           // 2^23 + 256 * 128
#pragma unroll
        for (int n1 = 0; n1 < 32; ++n1) {
            const int idx = M * (32 * n1 + lane) + r;
            const uint32_t v = in16[idx];
            const int q = bitrev<32>(n1);
            a[q] = cpack(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7504)),
                         __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7514)));
            if (WINDOW) {
                const float w = __ldg(&p.window[idx]);
                a[q] = cmul2(csub(a[q], bias1), cpack(w, w));
            }
        }
        fft1024_pass1<!WINDOW>(a);
    };
    gather_pass1(0);

    uint32_t f = 0;
    for (uint32_t it = 0; it < n_items; ++it) {
        const uint32_t item = blockIdx.x + it * gridDim.x;
        const size_t out_base = (size_t) item * N + (size_t) (r * MX_KPW * 32 + lane);
        for (int j = 0; j < K; ++j, ++f) {
            const int st = f % MX_STAGES;
            const int set = f & 1;
            float2* xch = reinterpret_cast<float2*>(tiles + (set * M + r) * FFT1024_XCH_BYTES);

            c64 b[32];
            fft1024_pass2(a, tw, xch, lane, b);
            // ---- Z_r[k] = W_N^(r k) F_r[k], k = lane + 32 k2, parked in this warp's tile as [k2][lane] ----
            __syncwarp();                         // every lane has finished reading the transpose
#pragma unroll
            for (int k2 = 0; k2 < 32; ++k2) {
                c64 z = b[k2];
                if (r > 0) {
                    const float2 w = __ldg(twr + 32 * k2);
                    z = cmul(z, w.x, w.y);
                }
                cstore(&reinterpret_cast<c64*>(xch)[k2 * 32 + lane], z);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&zfull[set]);
            if (f + 1 < n_frames) gather_pass1(f + 1);
            mbar_wait(&zfull[set], (f >> 1) & 1);
            if (tid == 0 && f + MX_STAGES < n_frames) {          // all branches have consumed the stage
                fence_proxy_async_smem();
                mbar_arrive_expect_tx(&full[st], MX_FRAME_BYTES);
                tma_load_1d(ring + st * MX_FRAME_BYTES, frame_src(f + MX_STAGES), MX_FRAME_BYTES, &full[st]);
            }

            // ---- combine: this warp owns k = (r * MX_KPW + g) * 32 + lane, g < MX_KPW ----
            const uint8_t* zset = tiles + set * M * FFT1024_XCH_BYTES;
            float pw[32];
#pragma unroll
            for (int g = 0; g < MX_KPW; ++g) {
                c64 z[M];
#pragma unroll
                for (int rr = 0; rr < M; ++rr)
                    z[bitrev<M>(rr)] =
                        reinterpret_cast<const c64*>(zset + rr * FFT1024_XCH_BYTES)[(r * MX_KPW + g) * 32 + lane];
                fft_dit_small<M>(z);
#pragma unroll
                for (int q = 0; q < M; ++q) {
                    float re, im;
                    cunpack(z[q], re, im);
                    pw[g * M + q] = fmaf(re, re, im * im);
                }
            }
            // spectrum.c:30-33: the DC position (bin 0: warp 0, g 0, q 0, lane 0) repeats its left neighbour,
            // bin N-1 = (k 1023, q M-1).  Warp 0 recomputes that one bin from the parked Z_r[1023] instead of
            // waiting for warp M-1 to hand it over.
            if (r == 0) {
                c64 z[M];
#pragma unroll
                for (int rr = 0; rr < M; ++rr)
                    z[bitrev<M>(rr)] = reinterpret_cast<const c64*>(zset + rr * FFT1024_XCH_BYTES)[1023];
                fft_dit_small<M>(z);
                float re, im;
                cunpack(z[M - 1], re, im);
                const float left = fmaf(re, re, im * im);
                if (MULTI) {
                    dcacc = fmaf((float) (K - j), left, dcacc);     // cumulative: sum_j (K - j) |X_j[N-1]|^2
                } else if (lane == 0) {
                    pw[0] = left;
                }
            }
            if (MULTI) {
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[i] += pw[i];
            } else {
                store_bins(p, dboff, out_base, pw);
            }
        }
        if (MULTI) {
            if (r == 0 && lane == 0) acc[0] = dcacc;
            store_bins(p, dboff, out_base, acc);
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
            dcacc = 0.0f;
        }
    }
}

}  // namespace

// N = 8192, cmplx_u8 input.  p.twiddle must be the 1024-point table and p.twiddle_n the [8][1024] table
// W_N^(r k) (capi.cu keeps both in the plan).
int launch_spectrum_mx1024(const SpecParams& p, cudaStream_t stream)
{
    const uint64_t total = (uint64_t) p.n_streams * (uint64_t) p.n_rows;
    auto kern = p.K > 1 ? (p.window ? spectrum_mx1024_kernel<true, true> : spectrum_mx1024_kernel<false, true>)
                        : (p.window ? spectrum_mx1024_kernel<true, false> : spectrum_mx1024_kernel<false, false>);
    if (int rc = ensure_dynamic_smem((const void*) kern, MX_SMEM)) return rc;
    const int ctas_per_sm = cached_occupancy((const void*) kern, MX_THREADS, MX_SMEM);
    uint64_t grid = (uint64_t) sm_count() * (uint64_t) ctas_per_sm;
    if (grid > total) grid = total;
    kern<<<(unsigned) grid, MX_THREADS, MX_SMEM, stream>>>(p);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

// spectrum1024.cu -- batched 1024-point power spectra, one warp per frame (sm_100a).
//
// Reference arithmetic reproduced per frame (paths relative to the reference's src/):
//   spectrum.c:54-58   unpack  in = (u8 - 128) / 128                (the /128 is folded into
//                                                                   the power scale: exact)
//   spectrum.c:21      unnormalised forward DFT (FFTW_FORWARD)
//   spectrum.c:23-34   out[i] += |X[(i + N/2) mod N]|^2, and out[N/2] += out[N/2 - 1]
//   cbb_main.c:125-128 10*log10(|g * P / K|), (int) truncation, clamp to [0, 255]
//
// Decomposition 1024 = 32 x 32 with n = 32*n1 + n2, k = k1 + 32*k2:
//   pass 1: lane n2 holds x[32*n1 + n2] (n1 = 0..31) in registers, 32-point FFT over n1,
//           multiply by W_1024^(n2*k1) (lane-private twiddles kept in registers for the
//           life of the persistent warp), write row k1 of a padded shared tile;
//   pass 2: lane k1 reads its row (all n2), 32-point FFT over n2 -> bins k1 + 32*k2.
// One shared-memory exchange per frame, warp-private: no block-level barrier anywhere.
// A warp store for fixed k2 covers 32 consecutive bins = 128 contiguous bytes.
//
// Input frames are staged by the TMA unit (cp.async.bulk, 2 KB per frame) into a
// warp-private two-deep ring guarded by mbarriers, so the next frame streams in from HBM
// while the current one is in the butterflies.
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

constexpr int N1024 = 1024;
constexpr int FRAME_BYTES = 2 * N1024;             // u8 re + u8 im
constexpr int XCH_BYTES = FFT1024_XCH_BYTES;
constexpr int WARP_SMEM = 2 * FRAME_BYTES + XCH_BYTES + 32;   // ring + exchange tile + 2 mbarriers (padded)
constexpr int WARPS_PER_CTA = 4;
constexpr float POWER_SCALE = FFT1024_POWER_SCALE;
constexpr int CTA_SMEM = WARPS_PER_CTA * WARP_SMEM + N1024 * 4;   // + window copy

// TMA producer cursor of one warp (only lane 0 uses it): walks the warp's rows, stride GW, and
// the K frames of each row, without a division per frame.
struct FrameCursor {
    uint32_t s, r, left;
    int j;
    __device__ __forceinline__ void init(const SpecParams& p, uint32_t item, uint32_t frames)
    {
        const uint32_t n_rows = (uint32_t) p.n_rows;
        s = item / n_rows;
        r = item - s * n_rows;
        j = 0;
        left = frames;
    }
    __device__ __forceinline__ const uint8_t* src(const SpecParams& p) const
    {
        return p.iq + (int64_t) s * p.stream_stride_bytes + 2 * ((int64_t) r * p.row_hop + (int64_t) j * p.hop);
    }
    __device__ __forceinline__ void advance(const SpecParams& p, int K, uint32_t GW)
    {
        --left;
        if (++j == K) {
            j = 0;
            r += GW;
            const uint32_t n_rows = (uint32_t) p.n_rows;
            while (r >= n_rows) {
                r -= n_rows;
                ++s;
            }
        }
    }
};

// pw[q] holds the raw power of bin lane + 32 * bitrev(q); write the requested outputs of one
// row in display order (fftshift = +16 on the k2 digit).  `base` = row * 1024 + lane, so every
// store is base + a compile-time offset and a warp store covers 128 contiguous bytes.
__device__ __forceinline__ void store_row(const SpecParams& p, float dboff, size_t base, const float (&pw)[32])
{
    if (p.db != nullptr) {
        float* out = p.db + base;
#pragma unroll
        for (int q = 0; q < 32; ++q)
            __stcs(out + fft1024_col(q), fmaf(DB_PER_LOG2, lg2_ftz(pw[q]), dboff));
    }
    if (p.power != nullptr) {
        float* out = p.power + base;
#pragma unroll
        for (int q = 0; q < 32; ++q) __stcs(out + fft1024_col(q), pw[q] * POWER_SCALE);
    }
    if (p.db_u8 != nullptr) {
        uint8_t* out = p.db_u8 + base;
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            // cbb_main.c:125-127: (int) truncation toward zero, then clamp; -inf / NaN -> 0
            int m = __float2int_rz(fmaf(DB_PER_LOG2, lg2_ftz(pw[q]), dboff));
            m = m < 0 ? 0 : (m > 255 ? 255 : m);
            out[fft1024_col(q)] = (uint8_t) m;
        }
    }
}

template <bool MULTI, bool WINDOW>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, MULTI ? 2 : 3) spectrum1024_kernel(const SpecParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    uint8_t* wbase = smem + warp * WARP_SMEM;
    uint8_t* ring = wbase;
    float2* xch = reinterpret_cast<float2*>(wbase + 2 * FRAME_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(wbase + 2 * FRAME_BYTES + XCH_BYTES);
    float* win = reinterpret_cast<float*>(smem + WARPS_PER_CTA * WARP_SMEM);

    if (WINDOW) {
        for (int i = threadIdx.x; i < N1024; i += blockDim.x) win[i] = p.window[i];
        __syncthreads();
    }

    const uint32_t total_items = (uint32_t) p.n_streams * (uint32_t) p.n_rows;
    const uint32_t gw = blockIdx.x * WARPS_PER_CTA + warp;
    const uint32_t GW = gridDim.x * WARPS_PER_CTA;
    if (gw >= total_items) return;
    const uint32_t n_items = (total_items - gw + GW - 1) / GW;
    const int K = MULTI ? p.K : 1;

    if (lane == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncwarp();

    float2 tw[32];
    fft1024_load_twiddles(p.twiddle, lane, tw);
    // the plan's offset folds gain, /K and 2^-14; the unpack's extra 256^2 goes here
    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;

    FrameCursor cur;
    cur.init(p, gw, n_items * (uint32_t) K);
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < 2; ++st) {
            if (cur.left > 0) {
                mbar_arrive_expect_tx(&bars[st], FRAME_BYTES);
                tma_load_1d(ring + st * FRAME_BYTES, cur.src(p), FRAME_BYTES, &bars[st]);
                cur.advance(p, K, GW);
            }
        }
    }

    float acc[32];
    float dcacc = 0.0f;
    if (MULTI) {
#pragma unroll
        for (int q = 0; q < 32; ++q) acc[q] = 0.0f;
    }

    uint32_t f = 0;
    for (uint32_t it = 0; it < n_items; ++it) {
        const uint32_t item = gw + it * GW;
        for (int j = 0; j < K; ++j, ++f) {
            const int st = f & 1;
            mbar_wait(&bars[st], (f >> 1) & 1);

            c64 a[32];
            fft1024_load<WINDOW>(reinterpret_cast<const uint16_t*>(ring + st * FRAME_BYTES), win, lane, a);
            __syncwarp();
            // stage `st` is free again: request the frame two ahead
            if (lane == 0 && cur.left > 0) {
                fence_proxy_async_smem();
                mbar_arrive_expect_tx(&bars[st], FRAME_BYTES);
                tma_load_1d(ring + st * FRAME_BYTES, cur.src(p), FRAME_BYTES, &bars[st]);
                cur.advance(p, K, GW);
            }
            float pw[32];
            fft1024_core<!WINDOW>(a, tw, xch, lane, pw);

            if (!MULTI) {
                // DC-position patch (spectrum.c:30-33): display index N/2 (bin 0: lane 0, q 0)
                // takes the value of display index N/2-1 (bin 1023: lane 31, q 31)
                const float left = __shfl_sync(0xffffffffu, pw[31], 31);
                if (lane == 0) pw[0] = left;
                store_row(p, dboff, (size_t) item * N1024 + lane, pw);
            } else {
#pragma unroll
                for (int q = 0; q < 32; ++q) acc[q] += pw[q];
                // cumulative DC patch: after K adds the DC position holds
                // sum_j (K - j) * |X_j[N-1]|^2, j = 0..K-1
                dcacc = fmaf((float) (K - j), pw[31], dcacc);
            }
        }
        if (MULTI) {
            const float left = __shfl_sync(0xffffffffu, dcacc, 31);
            if (lane == 0) acc[0] = left;
            store_row(p, dboff, (size_t) item * N1024 + lane, acc);
#pragma unroll
            for (int q = 0; q < 32; ++q) acc[q] = 0.0f;
            dcacc = 0.0f;
        }
    }
}

// ---- contiguous frames, K = 1 (BASELINE config 2: per-frame spectra of a long capture) ------------------
// When the frames of a stream follow each other without gap (hop = row_hop <= N, K = 1: contiguous or overlapping) the
// kernel above pays per frame for things that can be paid per six frames: one 2 KB TMA copy, one
// mbarrier round trip and a lane-0 cursor update per frame and warp.  This variant has the structure
// of chain_fused.cu without its FM branch: groups of six warps share a four-deep ring of 10 KB tiles
// (five consecutive frames, ONE bulk copy), full / empty mbarriers; per tile five warps transform a frame
// each and the sixth (rotating) only re-arms the ring; nobody meets at a block barrier, and one CTA per SM
// holds two such groups so that the twelve warps spread 3-3-3-3 over the schedulers.  Measured on the same
// data (256 streams x 8.192 M samples): 744 -> 787 Gsamples/s rectangular, 677 -> 738 Hann; with six frames
// per tile and all six warps transforming it is 785 / 721.
constexpr int T6_WARPS = 6;
constexpr int T6_GROUPS = 2;
constexpr int T6_THREADS = T6_GROUPS * T6_WARPS * 32;
constexpr int T6_STAGES = 4;
constexpr int T6_FRAMES = 5;                       // frames per tile: the sixth warp of the rotation only re-arms the ring
constexpr int T6_STAGE_BYTES = T6_FRAMES * FRAME_BYTES;
constexpr int T6_GROUP_SMEM = (T6_STAGES * T6_STAGE_BYTES + T6_WARPS * XCH_BYTES + 64 + 127) / 128 * 128;     // ring, tiles, 8 mbarriers (+pad)
static_assert(T6_GROUP_SMEM % 128 == 0, "group shared memory must keep the TMA destinations aligned");
constexpr int T6_SMEM = T6_GROUPS * T6_GROUP_SMEM + N1024 * 4;                        // + window copy

template <bool WINDOW>
__global__ void __launch_bounds__(T6_THREADS, 1) spectrum1024_tiled_kernel(const SpecParams p)
{
    extern __shared__ __align__(128) uint8_t smem_all[];
    const int lane = threadIdx.x & 31;
    const int group = (threadIdx.x >> 5) / T6_WARPS;
    const int warp = (threadIdx.x >> 5) % T6_WARPS;
    uint8_t* smem = smem_all + group * T6_GROUP_SMEM;
    uint8_t* ring = smem;
    float2* xch = reinterpret_cast<float2*>(smem + T6_STAGES * T6_STAGE_BYTES + warp * XCH_BYTES);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + T6_STAGES * T6_STAGE_BYTES + T6_WARPS * XCH_BYTES);
    uint64_t* empty = full + T6_STAGES;
    float* win = reinterpret_cast<float*>(smem_all + T6_GROUPS * T6_GROUP_SMEM);

    const uint32_t n_rows = (uint32_t) p.n_rows;
    const uint32_t tps = (n_rows + T6_FRAMES - 1) / T6_FRAMES;             // tiles per stream
    const uint32_t total_tiles = (uint32_t) p.n_streams * tps;
    const uint32_t first = blockIdx.x * T6_GROUPS + group;
    const uint32_t stride = gridDim.x * T6_GROUPS;
    const uint32_t n_mine = first < total_tiles ? (total_tiles - first + stride - 1) / stride : 0;

    auto issue = [&](uint32_t it) {
        const uint32_t tile = first + it * stride;
        const uint32_t s = tile / tps;
        const uint32_t t = tile - s * tps;
        const uint32_t frames = n_rows - t * T6_FRAMES < (uint32_t) T6_FRAMES ? n_rows - t * T6_FRAMES : (uint32_t) T6_FRAMES;
        const int st = it % T6_STAGES;
        // frames of a tile start `hop` samples apart (hop <= N: they may overlap) and arrive as one span
        const uint32_t bytes = 2u * ((frames - 1) * (uint32_t) p.hop + N1024);
        const uint8_t* src = p.iq + (int64_t) s * p.stream_stride_bytes + 2 * (int64_t) t * T6_FRAMES * p.hop;
        mbar_arrive_expect_tx(&full[st], bytes);
        tma_load_1d(ring + st * T6_STAGE_BYTES, src, bytes, &full[st]);
    };

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < T6_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], T6_WARPS);
        }
        fence_mbar_init();
        for (uint32_t it = 0; it < T6_STAGES - 1 && it < n_mine; ++it) issue(it);
    }
    if (WINDOW) {
        for (int i = threadIdx.x; i < N1024; i += blockDim.x) win[i] = p.window[i];
    }
    __syncthreads();

    float2 tw[32];
    fft1024_load_twiddles(p.twiddle, lane, tw);
    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;

    int service = 0;                      // which warp re-arms the ring for this tile: it mod 6
    for (uint32_t it = 0; it < n_mine; ++it) {
        const int st = it % T6_STAGES;
        const uint32_t tile = first + it * stride;
        const uint32_t s = tile / tps;
        const uint32_t t = tile - s * tps;
        int slot = warp - service - (T6_FRAMES < T6_WARPS ? 1 : 0);       // frames go to the other warps in rotation order
        if (slot < 0) slot += T6_WARPS;
        const uint32_t row = t * T6_FRAMES + slot;
        const bool serving_only = T6_FRAMES < T6_WARPS && warp == service;
        const bool have = row < n_rows && !serving_only;      // a short last tile leaves some warps without a frame

        mbar_wait(&full[st], (it / T6_STAGES) & 1);
        if (!serving_only) {
            c64 a[32];
            // (a warp without a frame transforms whatever its slot of the stage holds and stores nothing)
            fft1024_load<WINDOW>(reinterpret_cast<const uint16_t*>(ring + st * T6_STAGE_BYTES + 2 * p.hop * slot), win, lane, a);
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[st]);
                if (T6_FRAMES == T6_WARPS && warp == service && it + T6_STAGES - 1 < n_mine) {
                    if (it > 0) mbar_wait(&empty[(it - 1) % T6_STAGES], ((it - 1) / T6_STAGES) & 1);
                    fence_proxy_async_smem();
                    issue(it + T6_STAGES - 1);
                }
            }
            float pw[32];
            fft1024_core<!WINDOW>(a, tw, xch, lane, pw);
            // DC-position patch (spectrum.c:30-33): display index 512 takes display index 511's value
            const float left = __shfl_sync(0xffffffffu, pw[31], 31);
            if (lane == 0) pw[0] = left;
            if (have) {
                float* out = p.db + ((size_t) s * n_rows + row) * N1024 + lane;
#pragma unroll
                for (int q = 0; q < 32; ++q) __stcs(out + fft1024_col(q), fmaf(DB_PER_LOG2, lg2_ftz(pw[q]), dboff));
            }
        } else {
            if (lane == 0) {
                mbar_arrive(&empty[st]);
                // keep the ring full: tile it + STAGES - 1 goes into the stage tile it - 1 used
                if (it + T6_STAGES - 1 < n_mine) {
                    if (it > 0) mbar_wait(&empty[(it - 1) % T6_STAGES], ((it - 1) / T6_STAGES) & 1);
                    issue(it + T6_STAGES - 1);
                }
            }
            __syncwarp();
        }
        service = (service + 1 == T6_WARPS) ? 0 : service + 1;
    }
}

}  // namespace

int launch_spectrum1024(const SpecParams& p, cudaStream_t stream)
{
    const uint64_t total = (uint64_t) p.n_streams * (uint64_t) p.n_rows;
    const bool multi = p.K > 1;
    const bool window = p.window != nullptr;
    if (!multi && p.hop <= N1024 && p.row_hop == p.hop && p.n_rows >= 2 * T6_WARPS && p.db != nullptr && p.power == nullptr &&
        p.db_u8 == nullptr) {
        // frames hop <= N apart (contiguous or overlapping), dB rows only: five frames per TMA copy (tiles never span streams)
        auto tkern = window ? spectrum1024_tiled_kernel<true> : spectrum1024_tiled_kernel<false>;
        if (int rc = ensure_dynamic_smem((const void*) tkern, T6_SMEM)) return rc;
        const uint64_t tiles = (uint64_t) p.n_streams * (((uint64_t) p.n_rows + T6_FRAMES - 1) / T6_FRAMES);
        uint64_t tgrid = (uint64_t) sm_count();
        const uint64_t tneeded = (tiles + T6_GROUPS - 1) / T6_GROUPS;
        if (tgrid > tneeded) tgrid = tneeded;
        tkern<<<(unsigned) tgrid, T6_THREADS, T6_SMEM, stream>>>(p);
        B200_LAUNCH_CHECK();
        return B200_OK;
    }
    auto kern = multi ? (window ? spectrum1024_kernel<true, true> : spectrum1024_kernel<true, false>)
                      : (window ? spectrum1024_kernel<false, true> : spectrum1024_kernel<false, false>);
    if (int rc = ensure_dynamic_smem((const void*) kern, CTA_SMEM)) return rc;
    const int ctas_per_sm = cached_occupancy((const void*) kern, WARPS_PER_CTA * 32, CTA_SMEM);
    // persistent grid: a whole number of CTAs per SM, never more warps than rows
    uint64_t grid = (uint64_t) sm_count() * (uint64_t) ctas_per_sm;
    const uint64_t needed = (total + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    if (grid > needed) grid = needed;
    kern<<<(unsigned) grid, WARPS_PER_CTA * 32, CTA_SMEM, stream>>>(p);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

// fm_chain.cu -- the FM branch as ONE pass over the IQ bytes (sm_100a):
//   u8 IQ --CIC(R)--> int32 --atan2_approx--> phase --diff + limiter--> demod
//         --half-band /2--> --half-band /2--> float audio          (one float per 4R samples)
//
// Reference arithmetic (paths relative to the reference's src/): resample.c:6-45,
// common_sp.h:40-76, audio_main.c:110-139, resample.c:47-67.  The reference carries state
// in delay structs between 100 ms blocks; here every output is computed from its full
// dependency cone of INPUT samples instead -- audio[n] needs decimated samples 4n-31..4n,
// i.e. 32*R input samples of history -- so tiles are independent and the only state a
// stream carries between batches is its last 32*R input bytes pairs (b200sdr.h).
//
// A CTA walks tiles of T audio samples.  The tile's bytes ((4T + 32) * 2R, 10880 at
// R = 10) are staged by the TMA unit into a two-deep shared ring; phases:
//   1. one thread per decimated sample: byte sums with dp4a, atan2_approx, first difference
//      against the neighbour lane's phase (warp shuffle), limiter -> demod[] (smem)
//   2. one thread per first-stage output: half-band -> work[] (smem)
//   3. one thread per audio sample: half-band -> global
#include "b200_common.cuh"
#include "fm_kernels.cuh"

namespace b200 {

namespace {

constexpr int FM_THREADS = 256;

__host__ __device__ inline int fm_tile_audio(int R)
{
    int T = 128;
    while (T > 8 && (4 * T + 32) * 2 * R > 32768) T >>= 1;
    return T;
}

// One warp-wide step of the discriminator: lane handles local decimated index j (bytes at
// in + j * 2R); returns the phase (0 for j outside [0, nd)), and writes the CIC sums.
__device__ __forceinline__ float fm_phase_at(const uint8_t* in, int R, int j, int nd, int& sre, int& sim)
{
    uint32_t ure = CIC_MAGIC_BITS, uim = CIC_MAGIC_BITS;
    if (j >= 0 && j < nd) cic_sum(reinterpret_cast<const uint16_t*>(in) + (size_t) j * R, R, ure, uim);
    sre = (int) (ure - CIC_MAGIC_BITS);
    sim = (int) (uim - CIC_MAGIC_BITS);
    return atan2_approx_dev(__uint_as_float(uim) - CIC_MAGIC, __uint_as_float(ure) - CIC_MAGIC);
}

// Any R, sample-wise: the down factors 1, 2 and above 16 (3 <= R <= 16 take fm_chain_warp_kernel below).
__global__ void __launch_bounds__(FM_THREADS) fm_chain_kernel(const FmParams p, const int T, const int tiles_per_stream,
                                                              const int stage_bytes)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int R = p.R;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    uint8_t* ring = smem;
    float* demod = reinterpret_cast<float*>(smem + 2 * stage_bytes);      // d[j], local index as below
    float* work = demod + (4 * T + 32);
    uint64_t* bars = reinterpret_cast<uint64_t*>(work + (2 * T + 16));

    const int64_t n_audio = p.n_samples / (4 * R);
    const int64_t total_tiles = (int64_t) p.n_streams * tiles_per_stream;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto issue = [&](int64_t tile, int st) {
        const int s = (int) (tile / tiles_per_stream);
        const int64_t n0 = (int64_t) (tile - (int64_t) s * tiles_per_stream) * T;
        const int ta = (int) ((n_audio - n0) < T ? (n_audio - n0) : T);
        const uint32_t bytes = (uint32_t) (4 * ta + 32) * 2u * (uint32_t) R;
        const uint8_t* src = p.iq + (int64_t) s * p.stream_stride_bytes + (4 * n0 - 32) * 2 * (int64_t) R;
        mbar_arrive_expect_tx(&bars[st], bytes);
        tma_load_1d(ring + st * stage_bytes, src, bytes, &bars[st]);
    };

    int64_t tile = blockIdx.x;
    if (tid == 0) {
        if (tile < total_tiles) issue(tile, 0);
        if (tile + gridDim.x < total_tiles) issue(tile + gridDim.x, 1);
    }

    for (uint32_t it = 0; tile < total_tiles; tile += gridDim.x, ++it) {
        const int st = it & 1;
        const int s = (int) (tile / tiles_per_stream);
        const int64_t n0 = (int64_t) (tile - (int64_t) s * tiles_per_stream) * T;
        const int ta = (int) ((n_audio - n0) < T ? (n_audio - n0) : T);
        const int nd = 4 * ta + 32;       // decimated samples in this tile, local index 0 <-> 4*n0 - 32

        mbar_wait(&bars[st], (it >> 1) & 1);
        const uint8_t* in = ring + st * stage_bytes;

        // ---- phase 1: CIC boxcar (resample.c:21-40), atan2_approx, first difference and
        //      limiter (audio_main.c:110-131).  Lanes hold consecutive j, so phase[j-1] comes
        //      from the neighbour lane; lane 0 recomputes it. ----
        for (int j0 = (tid & ~31); j0 < nd; j0 += FM_THREADS) {
            const int j = j0 + lane;
            int sre, sim;
            const float ph = fm_phase_at(in, R, j, nd, sre, sim);
            float prev = __shfl_up_sync(0xffffffffu, ph, 1);
            if (lane == 0) {
                int a, b;
                prev = fm_phase_at(in, R, j - 1, nd, a, b);
            }
            if (j < nd) {
                demod[j] = fm_limit(ph, prev);
                if (p.decimated != nullptr && j >= 32) {
                    int2* dst = reinterpret_cast<int2*>(p.decimated) + (int64_t) s * p.dec_stride + (4 * n0 + (j - 32));
                    *dst = make_int2(sre, sim);
                }
            }
        }
        __syncthreads();
        // the input stage is consumed: refill it with the tile two steps ahead
        if (tid == 0) {
            const int64_t nxt = tile + 2 * (int64_t) gridDim.x;
            if (nxt < total_tiles) {
                fence_proxy_async_smem();
                issue(nxt, st);
            }
        }

        // ---- phase 2: half-band #1 (audio_main.c:133); work index 0 <-> 2*n0 - 10 ----
        const int nw = 2 * ta + 10;
        for (int m = tid; m < nw; m += FM_THREADS) work[m] = halfband_from(demod + 2 * m + 2);
        __syncthreads();

        // ---- phase 3: half-band #2 (audio_main.c:139) ----
        for (int a = tid; a < ta; a += FM_THREADS)
            p.audio[(int64_t) s * p.audio_stride + n0 + a] = halfband_from(work + 2 * a);
        // demod[] is rewritten by the next tile's phase 1 only after every thread has passed the
        // second __syncthreads above (all phase-2 reads done); work[] is rewritten in the next
        // tile's phase 2, after its first __syncthreads, which every phase-3 reader reaches first.
    }
}

// ---- 3 <= R <= 16 (R = 10 is the reference's default, cbb_main.c:80; its `bw` command gives
//      R = fs / 192000, main.c:154: 5 at 1.024, 12 at 2.4, 13 at 2.56, 15 at 2.88, 16 at 3.2 MS/s):
//      one WARP per tile, no block barriers ----
// Tile = 62 audio samples: 4*62 + 31 = 279 = 9 * 31 demodulator outputs, i.e. exactly nine
// shuffle chunks (lane 0 of a chunk only supplies the previous phase).  Input = (248 + 32) * R
// samples per TMA copy (5600 bytes at R = 10), two-deep warp-private ring; 13 KB of shared memory
// per warp at R = 10 (16 warps per SM).  Straight-line code: chunks that run past a short last tile
// read stale bytes of the ring and their results are simply not stored.
constexpr int FW_T = 62;
constexpr int FW_ND = 4 * FW_T + 32;              // 280 decimated samples, local index 0 <-> 4*n0 - 32
constexpr int FW_NW = 2 * FW_T + 10;              // 134 first-stage outputs

template <int R>
struct FwCfg {
    static constexpr int SAMPLE_BYTES = 2 * R;                     // one decimated sample's input
    static constexpr int STAGE = FW_ND * SAMPLE_BYTES;            // 5600 bytes at R = 10
    static constexpr int WARP_SMEM = 2 * STAGE + 288 * 4 + 144 * 4 + 32;   // ring, demod[], work[], 2 mbarriers (+pad)
    static_assert(WARP_SMEM % 16 == 0, "TMA destinations must stay 16-byte aligned");
    // warps per CTA: as many as let TWO CTAs share an SM (8 at R <= 10: 16 warps per SM; 7 at R = 12; 5 at R = 16)
    static constexpr int FIT = (113 * 1024) / WARP_SMEM;
    static constexpr int WARPS = FIT > 8 ? 8 : (FIT < 4 ? 4 : FIT);
    static constexpr int CTAS = 2;
};

template <int R>
__global__ void __launch_bounds__(FwCfg<R>::WARPS * 32, FwCfg<R>::CTAS) fm_chain_warp_kernel(const FmParams p, const int tiles_per_stream)
{
    using C = FwCfg<R>;
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    uint8_t* wbase = smem + warp * C::WARP_SMEM;
    uint8_t* ring = wbase;
    float* demod = reinterpret_cast<float*>(wbase + 2 * C::STAGE);
    float* work = demod + 288;
    uint64_t* bars = reinterpret_cast<uint64_t*>(work + 144);

    const int64_t n_audio = p.n_samples / (4 * R);
    const uint32_t tps = (uint32_t) tiles_per_stream;
    const uint32_t total_tiles = (uint32_t) p.n_streams * tps;
    const uint32_t gw = blockIdx.x * C::WARPS + warp;
    const uint32_t GW = gridDim.x * C::WARPS;
    if (gw >= total_tiles) return;
    const uint32_t n_mine = (total_tiles - gw + GW - 1) / GW;

    if (lane == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncwarp();

    auto issue = [&](uint32_t it) {
        const uint32_t tile = gw + it * GW;
        const uint32_t s = tile / tps;
        const int64_t n0 = (int64_t) (tile - s * tps) * FW_T;
        const int ta = (int) ((n_audio - n0) < FW_T ? (n_audio - n0) : FW_T);
        // (4 ta + 32) * 2R = 8 (ta + 8) R bytes from byte 8 (n0 - 8) R of the batch.  Both are multiples of 16:
        // n0 is a multiple of 62, and ta is even -- for odd R because n_samples = 4 R n_audio must be a multiple
        // of 8 (launch_fm_chain checks it), so n_audio and every n_audio - 62 k are even; for even R regardless.
        const uint32_t bytes = (uint32_t) (4 * ta + 32) * (uint32_t) C::SAMPLE_BYTES;
        const uint8_t* src = p.iq + (int64_t) s * p.stream_stride_bytes + (4 * n0 - 32) * C::SAMPLE_BYTES;
        const int st = it & 1;
        mbar_arrive_expect_tx(&bars[st], bytes);
        tma_load_1d(ring + st * C::STAGE, src, bytes, &bars[st]);
    };
    if (lane == 0) {
        issue(0);
        if (n_mine > 1) issue(1);
    }

    for (uint32_t it = 0; it < n_mine; ++it) {
        const int st = it & 1;
        const uint32_t tile = gw + it * GW;
        const uint32_t s = tile / tps;
        const int64_t n0 = (int64_t) (tile - s * tps) * FW_T;
        const int ta = (int) ((n_audio - n0) < FW_T ? (n_audio - n0) : FW_T);
        mbar_wait(&bars[st], (it >> 1) & 1);
        const uint8_t* in = ring + st * C::STAGE;

        // ---- discriminator: 9 chunks of 31 outputs (resample.c:21-40, common_sp.h:40-76,
        //      audio_main.c:110-131) ----
#pragma unroll
        for (int c = 0; c < 9; ++c) {
            const int j = 31 * c + lane;
            uint32_t ure, uim;
            if constexpr (R % 2 == 0)
                cic_even_sum<R>(reinterpret_cast<const uint32_t*>(in + j * C::SAMPLE_BYTES), ure, uim);
            else
                cic_odd_sum<R>(reinterpret_cast<const uint16_t*>(in + j * C::SAMPLE_BYTES), ure, uim);
            const float ph = atan2_approx_dev(__uint_as_float(uim) - CIC_MAGIC, __uint_as_float(ure) - CIC_MAGIC);
            const float prev = __shfl_up_sync(0xffffffffu, ph, 1);
            if (lane > 0) demod[j] = fm_limit(ph, prev);
            if (p.decimated != nullptr && j >= 32 && j < 4 * ta + 32) {
                int2* dst = reinterpret_cast<int2*>(p.decimated) + (int64_t) s * p.dec_stride + (4 * n0 + (j - 32));
                *dst = make_int2((int) (ure - CIC_MAGIC_BITS), (int) (uim - CIC_MAGIC_BITS));
            }
        }
        __syncwarp();
        if (lane == 0 && it + 2 < n_mine) {
            fence_proxy_async_smem();
            issue(it + 2);
        }
        // ---- half-band #1 (audio_main.c:133); work index 0 <-> 2*n0 - 10 ----
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            const int m = 32 * r + lane;
            if (m < FW_NW) work[m] = halfband_from(demod + 2 * m + 2);
        }
        __syncwarp();
        // ---- half-band #2 (audio_main.c:139) ----
        float* out = p.audio + (int64_t) s * p.audio_stride + n0;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int a = 32 * r + lane;
            if (a < ta) out[a] = halfband_from(work + 2 * a);
        }
        __syncwarp();       // demod[] / work[] are rewritten by the next tile
    }
}

template <int R>
int launch_fm_warp(const FmParams& p, cudaStream_t stream)
{
    using C = FwCfg<R>;
    const int64_t n_audio = p.n_samples / (4 * R);
    const int64_t tps = (n_audio + FW_T - 1) / FW_T;
    const int64_t total = (int64_t) p.n_streams * tps;
    if (total >= (1ll << 31)) {
        set_error("fm: batch too long");
        return B200_ERR_ARG;
    }
    const int smem = C::WARPS * C::WARP_SMEM;
    if (int rc = ensure_dynamic_smem((const void*) fm_chain_warp_kernel<R>, smem)) return rc;
    const int per_sm = cached_occupancy((const void*) fm_chain_warp_kernel<R>, C::WARPS * 32, smem);
    int64_t grid = (int64_t) sm_count() * per_sm;
    const int64_t needed = (total + C::WARPS - 1) / C::WARPS;
    if (grid > needed) grid = needed;
    fm_chain_warp_kernel<R><<<(unsigned) grid, C::WARPS * 32, smem, stream>>>(p, (int) tps);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

// history <- last H samples of the batch (per stream); H*2 bytes, 16-byte granules
__global__ void fm_history_carry_kernel(uint8_t* iq, int64_t stride, int n_streams, int64_t n_bytes, int hist_bytes)
{
    const int granules = hist_bytes / 16;
    const int64_t total = (int64_t) n_streams * granules;
    for (int64_t i = blockIdx.x * (int64_t) blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x) {
        const int s = (int) (i / granules);
        const int g = (int) (i - (int64_t) s * granules);
        uint8_t* base = iq + (int64_t) s * stride;
        const uint4 v = *reinterpret_cast<const uint4*>(base + n_bytes - hist_bytes + 16 * g);
        *reinterpret_cast<uint4*>(base - hist_bytes + 16 * g) = v;
    }
}

__global__ void fm_history_reset_kernel(uint8_t* iq, int64_t stride, int n_streams, int hist_bytes)
{
    const int granules = hist_bytes / 16;
    const int64_t total = (int64_t) n_streams * granules;
    const uint4 v = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
    for (int64_t i = blockIdx.x * (int64_t) blockDim.x + threadIdx.x; i < total; i += (int64_t) gridDim.x * blockDim.x) {
        const int s = (int) (i / granules);
        const int g = (int) (i - (int64_t) s * granules);
        *reinterpret_cast<uint4*>(iq + (int64_t) s * stride - hist_bytes + 16 * g) = v;
    }
}

}  // namespace

int fm_history_samples(int R)
{
    return 32 * R;
}

int launch_fm_chain(const FmParams& p, cudaStream_t stream)
{
    if (p.R < 1 || p.R > 256) {
        set_error("fm: down factor %d outside [1, 256]", p.R);
        return B200_ERR_ARG;
    }
    if (p.n_samples < 0 || p.n_samples % (4 * p.R) != 0 || p.n_samples % 8 != 0) {
        set_error("fm: n_samples %lld must be a multiple of 4*R and of 8", (long long) p.n_samples);
        return B200_ERR_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(p.iq) & 15) != 0 || (p.stream_stride_bytes & 15) != 0) {
        set_error("fm: IQ pointer and stream stride must be 16-byte aligned");
        return B200_ERR_ALIGN;
    }
    if (p.n_streams == 0 || p.n_samples == 0) return B200_OK;
    switch (p.R) {                                  // small down factors: the warp-per-tile kernel
        case 3: return launch_fm_warp<3>(p, stream);
        case 5: return launch_fm_warp<5>(p, stream);
        case 7: return launch_fm_warp<7>(p, stream);
        case 9: return launch_fm_warp<9>(p, stream);
        case 11: return launch_fm_warp<11>(p, stream);
        case 13: return launch_fm_warp<13>(p, stream);
        case 15: return launch_fm_warp<15>(p, stream);
        case 4: return launch_fm_warp<4>(p, stream);
        case 6: return launch_fm_warp<6>(p, stream);
        case 8: return launch_fm_warp<8>(p, stream);
        case 10: return launch_fm_warp<10>(p, stream);
        case 12: return launch_fm_warp<12>(p, stream);
        case 14: return launch_fm_warp<14>(p, stream);
        case 16: return launch_fm_warp<16>(p, stream);
        default: break;
    }
    const int T = fm_tile_audio(p.R);
    const int64_t n_audio = p.n_samples / (4 * p.R);
    const int64_t tiles_per_stream = (n_audio + T - 1) / T;
    if (tiles_per_stream >= (1ll << 31)) {
        set_error("fm: batch too long");
        return B200_ERR_ARG;
    }
    const int stage_bytes = (4 * T + 32) * 2 * p.R;
    const int smem = 2 * stage_bytes + (4 * T + 32) * 4 + (2 * T + 16) * 4 + 16;
    if (int rc = ensure_dynamic_smem((const void*) fm_chain_kernel, 2 * 32768 + 8192)) return rc;
    const int ctas_per_sm = cached_occupancy((const void*) fm_chain_kernel, FM_THREADS, smem);
    int64_t grid = (int64_t) sm_count() * ctas_per_sm;
    const int64_t total_tiles = (int64_t) p.n_streams * tiles_per_stream;
    if (grid > total_tiles) grid = total_tiles;
    fm_chain_kernel<<<(unsigned) grid, FM_THREADS, smem, stream>>>(p, T, (int) tiles_per_stream, stage_bytes);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

// History of any length (a positive multiple of 8 samples): the FM chain's 32 R, or the longer one a channel FIR
// reaches back over (fm_channels_fir.cu)
int launch_iq_history_carry(uint8_t* iq, int64_t stride, int n_streams, int64_t n_samples, int hist_samples,
                            cudaStream_t stream)
{
    const int hist_bytes = 2 * hist_samples;
    if (n_samples * 2 < hist_bytes) {
        set_error("fm: batch shorter than the history (%d samples)", hist_samples);
        return B200_ERR_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(iq) & 15) != 0 || (stride & 15) != 0 || ((n_samples * 2) & 15) != 0) {
        set_error("fm history carry: pointer, stride and batch bytes must be multiples of 16");
        return B200_ERR_ALIGN;
    }
    if (n_streams == 0) return B200_OK;
    const int64_t total = (int64_t) n_streams * (hist_bytes / 16);
    const int blocks = (int) ((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    fm_history_carry_kernel<<<blocks, 256, 0, stream>>>(iq, stride, n_streams, n_samples * 2, hist_bytes);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

int launch_iq_history_reset(uint8_t* iq, int64_t stride, int n_streams, int hist_samples, cudaStream_t stream)
{
    const int hist_bytes = 2 * hist_samples;
    if ((reinterpret_cast<uintptr_t>(iq) & 15) != 0 || (stride & 15) != 0) {
        set_error("fm history reset: pointer and stride must be multiples of 16");
        return B200_ERR_ALIGN;
    }
    if (n_streams == 0) return B200_OK;
    const int64_t total = (int64_t) n_streams * (hist_bytes / 16);
    const int blocks = (int) ((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    fm_history_reset_kernel<<<blocks, 256, 0, stream>>>(iq, stride, n_streams, hist_bytes);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

int IqRows::alloc(int hist_samples, cudaStream_t stream)
{
    hist = hist_samples;
    pitch = 2 * ((int64_t) hist + max_batch);
    B200_CUDA_TRY(cudaMalloc((void**) &d_base, (size_t) n_rows * (size_t) pitch));
    return reset(stream);
}

int IqRows::create(int R_, int n_rows_, int64_t max_batch_, cudaStream_t stream)
{
    R = R_;
    n_rows = n_rows_;
    max_batch = max_batch_;
    return alloc(fm_history_samples(R), stream);
}

void IqRows::free()
{
    cudaFree(d_base);
    cudaFree(d_taps);
    d_base = nullptr;
    d_taps = nullptr;
    n_taps = 0;
}

int IqRows::reset(cudaStream_t stream)
{
    if (int rc = launch_iq_history_reset(batch(0), pitch, n_rows, hist, stream)) return rc;
    B200_CUDA_TRY(cudaStreamSynchronize(stream));
    return B200_OK;
}

int IqRows::carry(int i0, int n, int64_t n_samples, cudaStream_t stream)
{
    return launch_iq_history_carry(batch(i0), pitch, n, n_samples, hist, stream);
}

}  // namespace b200

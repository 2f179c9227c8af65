// chain_fused.cu -- the full chain in ONE pass over the IQ bytes (sm_100a): per-frame
// 1024-point dB spectra (K = 1, rectangular: spectrum.c + cbb_main.c:125) and the FM branch
// at R = 10 (resample.c, common_sp.h:40-76, audio_main.c:110-139) from the same shared-memory
// copy of the samples, so HBM sees each input byte once: 2 B in + 4 B dB + 0.1 B audio per
// sample, the algorithmic minimum (SURVEY.md section 8d).
//
// Tile = 5120 samples = lcm(1024, 4 * 10): 5 frames and 128 audio samples, plus the FM
// branch's 320-sample history (32 decimated samples) in front: 10880 bytes, fetched by one
// TMA bulk copy into a four-deep ring with full/empty mbarriers.  A tile is six jobs:
//   - five frame jobs: 3 of the tile's 18 discriminator chunks (CIC sums with dp4a,
//     atan2_approx, difference + limiter -> demod[], four buffers deep), then unpack one frame
//     into registers, release the stage, run the 32x32 two-pass transform, |X|^2, dB and store
//     4 KB of spectrum;
//   - one service job: 3 chunks, re-arm the TMA producer and run the two half-band decimators
//     of the PREVIOUS tile -> 128 audio floats.
// One CTA per SM of 18 warps; each warp takes the next job from a shared counter, so no warp is
// tied to a role and none meets another at a block barrier between set-up and exit.  The
// inter-pass twiddles come from a table in tensor memory (64 columns of every lane, filled once at
// kernel start), read 16 columns at a time just before pass 2's first stage uses them: not 62
// registers per lane, which would rule out 18 warps, and not shared memory, whose pipe the
// transpose already keeps busy.
// Tiles are independent (a tile's audio depends on input bytes only, through the history), so
// CTAs stride over (stream, tile) with no inter-CTA communication.
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "fm_kernels.cuh"

namespace b200 {

namespace {

constexpr int CF_WARPS = 18;
constexpr int CF_THREADS = CF_WARPS * 32;
constexpr int CF_STAGES = 4;                        // TMA ring
constexpr int CF_DBUF = 4;                          // demod[] / work[] buffers: tiles a fast warp may run ahead
constexpr int CF_TILE = 5120;                       // samples
constexpr int CF_HIST = 320;                        // samples of history in front of a tile
constexpr int CF_STAGE_BYTES = 2 * (CF_TILE + CF_HIST);   // 10880
constexpr int CF_ND_PAD = 576;                      // demod[] pitch: 544 decimated samples per tile, but the
                                                    // 18 chunks of 31 cover indices up to 557
constexpr int CF_NW = 2 * 128 + 10;                 // 266 first-stage outputs per tile
constexpr int CF_WORK = 272;                        // CF_NW padded

constexpr int CF_RING_BYTES = CF_STAGES * CF_STAGE_BYTES;
constexpr int CF_XCH_BYTES = CF_WARPS * FFT1024_XCH_BYTES;
constexpr int CF_DEMOD_BYTES = CF_DBUF * CF_ND_PAD * 4;
constexpr int CF_WORK_BYTES = CF_DBUF * CF_WORK * 4;
constexpr int CF_BAR_BYTES = (2 * CF_STAGES + 2 * CF_DBUF) * 8 + 8;     // + the job counter and the TMEM base
constexpr int CF_SMEM = CF_RING_BYTES + CF_XCH_BYTES + CF_DEMOD_BYTES + CF_WORK_BYTES + CF_BAR_BYTES;
static_assert(CF_SMEM <= 232448, "more shared memory than a CTA may have on sm_100");
static_assert(CF_STAGE_BYTES % 128 == 0, "ring stages must stay 128-byte aligned");
// A waiter tests the PARITY of a barrier phase, so it must never get two phases ahead of the barrier: no job of
// tile it + S (or it + D) may be claimed while a job of tile it is still running.  Jobs are claimed in order and
// at most W are in flight, so the first job of tile it + S (number 6 (it + S)) is claimed after job
// 6 (it + S) - W + 1 - 1 has been claimed and ... finished only if it is older than every running job:
// 6 (it + S) - (W - 1) > 6 it + 5.  (W = 20, S = 3 broke exactly this at kernel start: measured, 78 dB off.)
static_assert(CF_WARPS <= 6 * CF_STAGES - 5, "ring too shallow for this many warps: a full[] waiter could lap the barrier");
// demod[] buffers: the audio job of tile it (job 6 (it + 1)) waits for phase it / D of demod_full[it % D]; it would
// pass a phase early if the audio job of tile it - D (6 D jobs older) had not passed its own wait yet
static_assert(CF_WARPS <= 6 * CF_DBUF, "too few demod buffers for this many warps");

struct ChainParams {
    const uint8_t* iq;             // stream 0, first sample of the batch (history lies before it)
    int64_t stream_stride_bytes;
    int n_streams;
    int tiles_per_stream;
    float* db;                     // [n_streams][tiles_per_stream * 5][1024]
    float* audio;                  // [n_streams][tiles_per_stream * 128], row stride audio_stride
    int64_t audio_stride;
    float dboff;                   // 10*log10(g) + FFT1024_DB_SHIFT
    uint32_t tps_magic;            // tile / tiles_per_stream = (tile * tps_magic) >> tps_shift for tile < 2^31
    int tps_shift;
    const float2* twiddle;
};

// The six jobs of a tile (service + five frames) are not tied to particular warps: every warp takes the next job
// from a shared counter, and a warp that drew the short service job simply comes back sooner.  Jobs are claimed in
// order and only ever wait for lower-numbered jobs (ring refills, demod hand-off), so the lowest unfinished job can
// always run: no deadlock whatever the interleaving.  The inter-pass twiddles W_1024^(n2 k1) come from tensor
// memory: warps 0-3 write the same table into the four lane quadrants (lane k1 of a quadrant holds what lane k1 of a
// warp needs, see fft1024_pass2_tmem_tw), and every warp reads its quadrant with four tcgen05.ld per frame.
__global__ void __launch_bounds__(CF_THREADS, 1) chain_jobs_kernel(const ChainParams p)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    uint8_t* ring = smem;
    float2* xch = reinterpret_cast<float2*>(smem + CF_RING_BYTES + warp * FFT1024_XCH_BYTES);
    float* demod_base = reinterpret_cast<float*>(smem + CF_RING_BYTES + CF_XCH_BYTES);         // [CF_DBUF][CF_ND_PAD]
    float* work_base = demod_base + CF_DBUF * CF_ND_PAD;                                         // [CF_DBUF][CF_WORK]
    uint64_t* full = reinterpret_cast<uint64_t*>(work_base + CF_DBUF * CF_WORK);
    uint64_t* empty = full + CF_STAGES;
    uint64_t* demod_full = empty + CF_STAGES;
    uint64_t* demod_empty = demod_full + CF_DBUF;
    uint32_t* next_job = reinterpret_cast<uint32_t*>(demod_empty + CF_DBUF);
    uint32_t* tmem_slot = next_job + 1;

    const uint32_t total_tiles = (uint32_t) p.n_streams * (uint32_t) p.tiles_per_stream;
    const uint32_t first = blockIdx.x;
    const uint32_t stride = gridDim.x;
    const uint32_t n_mine = first < total_tiles ? (total_tiles - first + stride - 1) / stride : 0;

    // tile -> (stream, tile in stream) without a division: tile * magic >> shift (exact below 2^31)
    auto locate = [&](uint32_t tile, uint32_t& s, uint32_t& t) {
        s = (uint32_t) (((uint64_t) tile * p.tps_magic) >> p.tps_shift);
        t = tile - s * (uint32_t) p.tiles_per_stream;
    };
    auto issue = [&](uint32_t it) {
        uint32_t s, t;
        locate(first + it * stride, s, t);
        const int st = it % CF_STAGES;
        const uint8_t* src = p.iq + (int64_t) s * p.stream_stride_bytes + 2 * ((int64_t) t * CF_TILE - CF_HIST);
        mbar_arrive_expect_tx(&full[st], CF_STAGE_BYTES);
        tma_load_1d(ring + st * CF_STAGE_BYTES, src, CF_STAGE_BYTES, &full[st]);
    };
    // the two half-band decimators of local tile `it` (audio_main.c:133,139); one warp
    auto audio_job = [&](uint32_t it) {
        uint32_t s, t;
        locate(first + it * stride, s, t);
        const int buf = it % CF_DBUF;
        const float* demod = demod_base + buf * CF_ND_PAD;
        float* work = work_base + buf * CF_WORK;
        mbar_wait(&demod_full[buf], (it / CF_DBUF) & 1);
        for (int m = lane; m < CF_NW; m += 32)              // work index 0 <-> 2*n0 - 10
            work[m] = halfband_from(demod + 2 * m + 2);
        __syncwarp();
        if (lane == 0) mbar_arrive(&demod_empty[buf]);
        float* out = p.audio + (int64_t) s * p.audio_stride + (int64_t) t * 128;
#pragma unroll
        for (int r = 0; r < 4; ++r) out[32 * r + lane] = halfband_from(work + 2 * (32 * r + lane));
    };

    if (warp == 0) tmem_alloc(tmem_slot, FFT1024_TMEM_COLS);
    if (warp == 0 && lane == 0) {
        for (int i = 0; i < CF_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 6);
        }
        for (int i = 0; i < CF_DBUF; ++i) {
            mbar_init(&demod_full[i], 6);
            mbar_init(&demod_empty[i], 1);
        }
        *next_job = 0;
        fence_mbar_init();
        for (uint32_t it = 0; it < CF_STAGES - 1 && it < n_mine; ++it) issue(it);
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tw_taddr = *tmem_slot + ((uint32_t) (32 * (warp % 4)) << 16);     // this warp's quadrant
    if (warp < 4) {
#pragma unroll 1
        for (int c = 0; c < FFT1024_TMEM_COLS / FFT1024_TMEM_CHUNK; ++c) {
            uint32_t r[FFT1024_TMEM_CHUNK];
            fft1024_tmem_twiddles(p.twiddle, lane, c, r);
            tmem_st_32x32b_x16(tw_taddr + FFT1024_TMEM_CHUNK * c, r);
        }
        tmem_wait_st();
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();

    // jobs 6*it + pos: pos 0 = the tile's service job, 1..5 = frames 0..4; job 6*n_mine = the last tile's audio
    const uint32_t n_jobs = n_mine > 0 ? 6 * n_mine + 1 : 0;
    for (;;) {
        uint32_t job = 0;
        if (lane == 0) job = atomicAdd(next_job, 1u);
        job = __shfl_sync(0xffffffffu, job, 0);
        if (job >= n_jobs) break;
        const uint32_t it = job / 6;
        const int pos = (int) (job - 6 * it);
        if (it == n_mine) {
            audio_job(n_mine - 1);
            break;
        }
        const int st = it % CF_STAGES;
        const int buf = it % CF_DBUF;
        float* demod = demod_base + buf * CF_ND_PAD;

        mbar_wait(&full[st], (it / CF_STAGES) & 1);
        const uint8_t* in = ring + st * CF_STAGE_BYTES;

        // ---- discriminator share: 3 of the tile's 18 chunks of 31 outputs (lane 0 only supplies
        //      phase[j-1]); demod[buf] must have been drained by the audio job of tile it - CF_DBUF ----
        if (it >= (uint32_t) CF_DBUF) mbar_wait(&demod_empty[buf], ((it / CF_DBUF) - 1) & 1);
#pragma unroll
        for (int c3 = 0; c3 < 3; ++c3) {
            const int j = 31 * (pos + 6 * c3) + lane;
            // the last chunk's lanes 17..31 read up to 280 bytes past the stage -- still inside this
            // CTA's shared memory -- and write demod[544..557], padding that is never read
            uint32_t ure, uim;
            cic10_sum(reinterpret_cast<const uint32_t*>(in + j * 20), ure, uim);
            const float ph = atan2_approx_dev2(__uint_as_float(uim) - CIC_MAGIC, __uint_as_float(ure) - CIC_MAGIC);
            const float prev = __shfl_up_sync(0xffffffffu, ph, 1);
            if (lane > 0) demod[j] = fm_limit(ph, prev);                   // demod[0] is never read
        }

        if (pos > 0) {
            const int slot = pos - 1;
            c64 a[32];
            fft1024_load<false>(reinterpret_cast<const uint16_t*>(in + 2 * CF_HIST + 2048 * slot), nullptr, lane, a);
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[st]);
                mbar_arrive(&demod_full[buf]);
            }
            fft1024_pass1<true>(a);
            c64 b[32];
            fft1024_pass2_tmem_tw(a, tw_taddr, xch, lane, b);
            float pw[32];
            fft1024_power(b, pw);
            // DC-position patch (spectrum.c:30-33): display index 512 takes display index 511's value
            const float left = __shfl_sync(0xffffffffu, pw[31], 31);
            if (lane == 0) pw[0] = left;
            // rows of all streams are contiguous: row = 5 * tile + frame
            fft1024_store_db(p.db + ((size_t) (first + it * stride) * 5 + slot) * 1024 + lane, pw, p.dboff);
        } else {
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[st]);
                mbar_arrive(&demod_full[buf]);
                // keep the ring full: tile it + CF_STAGES - 1 goes into the stage tile it - 1 used
                if (it + CF_STAGES - 1 < n_mine) {
                    if (it > 0) mbar_wait(&empty[(it - 1) % CF_STAGES], ((it - 1) / CF_STAGES) & 1);
                    issue(it + CF_STAGES - 1);
                }
            }
            __syncwarp();
            if (it > 0) audio_job(it - 1);
        }
    }

    // every warp's last tcgen05.ld has completed (each pass 2 waits for its loads) before the table is freed
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tmem_fence_after_sync();
        tmem_dealloc(*tmem_slot, FFT1024_TMEM_COLS);     // read again: a register held over the job loop costs more
        tmem_relinquish_alloc_permit();
    }
}

}  // namespace

int launch_chain_fused(const uint8_t* d_iq, int64_t stride, int n_streams, int64_t n_samples, float db_offset,
                       const float2* twiddle, float* d_db, float* d_audio, int64_t audio_stride, cudaStream_t stream)
{
    const int64_t tiles_per_stream = n_samples / CF_TILE;
    const int64_t total = (int64_t) n_streams * tiles_per_stream;
    if (total == 0) return B200_OK;
    if (total >= (1ll << 31) || tiles_per_stream * 5 * 1024 >= (1ll << 40)) {
        set_error("chain: too many tiles in one launch (%lld)", (long long) total);
        return B200_ERR_ARG;
    }
    ChainParams p;
    p.iq = d_iq;
    p.stream_stride_bytes = stride;
    p.n_streams = n_streams;
    p.tiles_per_stream = (int) tiles_per_stream;
    p.db = d_db;
    p.audio = d_audio;
    p.audio_stride = audio_stride;
    // the plan's offset is 10*log10(g / (K * 2^14)) with K = 1; the fused unpack carries 2^30
    p.dboff = db_offset - 16.0f * DB_PER_LOG2;
    p.twiddle = twiddle;
    // tile / tiles_per_stream by multiplication: L = ceil(log2 d), magic = ceil(2^(31+L) / d) fits 32 bits and is
    // exact for every tile < 2^31 (the error magic * d - 2^(31+L) is below d <= 2^L)
    int L = 0;
    while ((1ll << L) < tiles_per_stream) ++L;
    p.tps_magic = (uint32_t) (((1ull << (31 + L)) + (uint64_t) tiles_per_stream - 1) / (uint64_t) tiles_per_stream);
    p.tps_shift = 31 + L;
    if (int rc = ensure_dynamic_smem((const void*) chain_jobs_kernel, CF_SMEM)) return rc;
    int64_t grid = sm_count();
    if (grid > total) grid = total;
    chain_jobs_kernel<<<(unsigned) grid, CF_THREADS, CF_SMEM, stream>>>(p);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

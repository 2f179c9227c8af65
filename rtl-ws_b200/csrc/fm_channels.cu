// fm_channels.cu -- several FM channels at frequency offsets inside one dongle's band, one pass over the IQ
// bytes for all channels of a stream (sm_100a).
//
// Channel c of stream s has a 32-bit phase increment inc (b200_fm_channel_tune).  Sample n (int64, from stream
// start; the history has n < 0) is mixed with exp(-j 2 pi phi(n) / 2^32), phi(n) = (uint32)(inc * (uint64) n),
// then the reference's boxcar (resample.c:21-40, no 1/128) and demodulator (audio_main.c:110-139) follow:
//   b[m] = sum_{k<R} x[mR + k] exp(-j phi(mR + k))  =  exp(-j phi(mR)) * sum_{k<R} x[mR + k] w[k],
//   w[k] = exp(-j 2 pi inc k / 2^32)
// because phi(mR + k) = phi(mR) + phi(k) exactly mod 2^32.  So the mixer plus boxcar is an R-tap complex filter
// per channel followed by ONE rotation per decimated sample, whose angle comes from the exact integer phase of
// sample mR (never from a running float phase, which would drift over a long stream).  At inc = 0 the taps are
// (1, 0) and every rotation is (1, 0) exactly, so b is the integer CIC output and the audio is b200_fm_exec's.
//
// Geometry: the tile of fm_chain_warp_kernel (62 audio samples = 4*62 + 32 decimated samples, 9 shuffle chunks of
// 31 demodulator outputs), staged by the TMA into a ring of the CTA.  One CTA of 9 warps per tile, one warp per
// chunk, so no lane is idle in the discriminator.  Channels are handled G at a time:
//   0. taps w[g][k] of the group (accurate sincospif of the exact integer phase) -> smem
//   1. warp = chunk, lane = decimated sample: complex MAC over the R input samples (packed f32x2 FMAs), rotation,
//      atan2_approx, first difference against the neighbour lane, limiter -> demod[g][] (smem)
//   2. half-band #1 -> work[g][] (smem)          3. half-band #2 -> audio row s*C + c
// At R = 10 a lane unpacks its ten byte pairs into registers once per tile and reuses them for every channel;
// any other R reads and unpacks the bytes once per channel.
#include <string.h>

#include "b200_common.cuh"
#include "fm_channels.cuh"
#include "fm_kernels.cuh"

namespace b200 {

namespace {

// The tile loop of both forms.  RUNS: p is an FcRunsParams, p.n_streams counts runs, and each tile takes its IQ
// row, channel count, increments, position and audio rows from its run; no baseband.  The channel loop bound is the
// tile's, the same for every thread of the CTA, so the three barriers per group stay uniform.
template <int RT, int G, bool RUNS, class P>
__device__ __forceinline__ void fm_channels_tiles(const P& p, const int tiles_per_stream, const int stage_bytes,
                                                  const int n_stages)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int R = RT ? RT : p.R;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    uint8_t* ring = smem;
    float4* taps = reinterpret_cast<float4*>(smem + n_stages * stage_bytes);   // [G][R]: (w.re, w.im, -w.im, w.re)
    float* demod = reinterpret_cast<float*>(taps + G * R);                        // [G][FC_DEMOD]
    float* work = demod + G * FC_DEMOD;                                           // [G][FC_WORK]
    uint64_t* bars = reinterpret_cast<uint64_t*>(work + G * FC_WORK);

    const int C_all = p.n_channels;
    const int64_t n_audio = p.n_samples / (4 * R);
    const int64_t total_tiles = (int64_t) p.n_streams * tiles_per_stream;
    const uint32_t first_dec_all = (uint32_t) (p.first_sample / R);      // mod 2^32, like every phase below

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto issue = [&](int64_t tile, int st) {
        const int q = (int) (tile / tiles_per_stream);
        const int s = RUNS ? fc_run<RUNS>(p, q)->stream : q;
        const int64_t n0 = (tile - (int64_t) q * tiles_per_stream) * FC_T;
        const int ta = (int) ((n_audio - n0) < FC_T ? (n_audio - n0) : FC_T);
        // 8 (ta + 8) R bytes from byte 8 (n0 - 8) R: multiples of 16 (n0 is a multiple of 62; ta is even for odd R
        // because n_samples is a multiple of 8 and of 4R), as in fm_chain_warp_kernel
        const uint32_t bytes = (uint32_t) (4 * ta + 32) * 2u * (uint32_t) R;
        const uint8_t* src = p.iq + (int64_t) s * p.stream_stride_bytes + (4 * n0 - 32) * 2 * (int64_t) R;
        mbar_arrive_expect_tx(&bars[st], bytes);
        tma_load_1d(ring + st * stage_bytes, src, bytes, &bars[st]);
    };

    int64_t tile = blockIdx.x;
    if (tid == 0)
        for (int k = 0; k < n_stages; ++k)
            if (tile + k * (int64_t) gridDim.x < total_tiles) issue(tile + k * (int64_t) gridDim.x, k);

    for (uint32_t it = 0; tile < total_tiles; tile += gridDim.x, ++it) {
        const int st = (int) (it % (uint32_t) n_stages);
        const int q = (int) (tile / tiles_per_stream);
        // the runs form: this tile's IQ row, channel count, position, increments and audio rows come from its run
        const FcRun* run = fc_run<RUNS>(p, q);
        const int s = RUNS ? run->stream : q;
        const int C = RUNS ? run->n_channels : C_all;
        const uint32_t first_dec = RUNS ? run->first_dec : first_dec_all;
        const int64_t n0 = (tile - (int64_t) q * tiles_per_stream) * FC_T;
        const int ta = (int) ((n_audio - n0) < FC_T ? (n_audio - n0) : FC_T);
        const int j = 31 * warp + lane;                                   // this lane's decimated sample
        const uint32_t m = first_dec + (uint32_t) (4 * n0 - 32) + (uint32_t) j;
        const uint32_t* incs = RUNS ? run->phase_inc : p.phase_inc + (int64_t) s * C;

        mbar_wait(&bars[st], (it / (uint32_t) n_stages) & 1);
        const uint8_t* in = ring + st * stage_bytes + j * 2 * R;

        // R = 10: the lane's ten samples unpacked once per tile, as duplicated pairs (re, re) and (im, im)
        c64 xr[RT ? RT : 1], xi[RT ? RT : 1];
        if constexpr (RT == 10) {
#pragma unroll
            for (int w = 0; w < 5; ++w) {
                const uint32_t v = reinterpret_cast<const uint32_t*>(in)[w];
                xr[2 * w] = byte_pair(v, 0);
                xi[2 * w] = byte_pair(v, 1);
                xr[2 * w + 1] = byte_pair(v, 2);
                xi[2 * w + 1] = byte_pair(v, 3);
            }
        }

        for (int c0 = 0; c0 < C; c0 += G) {
            const int gc = (C - c0) < G ? (C - c0) : G;
            // ---- 0. taps of the group ----
            for (int i = tid; i < gc * R; i += FC_THREADS) {
                const int g = i / R, k = i - g * R;
                const uint32_t phi = incs[c0 + g] * (uint32_t) k;
                float sn, cs;
                sincospif((float) (int32_t) phi * 4.65661287307739258e-10f, &sn, &cs);     // 2^-31: [-1, 1)
                taps[g * R + k] = make_float4(cs, -sn, sn, cs);
            }
            __syncthreads();

            // ---- 1. mix + boxcar, rotation, discriminator (common_sp.h:40-76, audio_main.c:110-131) ----
#pragma unroll
            for (int g = 0; g < G; ++g) {
                if (g < gc) {
                    const float4* w = taps + g * R;
                    c64 acc = cpack(0.0f, 0.0f);
                    if constexpr (RT == 10) {
#pragma unroll
                        for (int k = 0; k < RT; ++k) {
                            const float4 t = w[k];
                            acc = cfma2(xr[k], cpack(t.x, t.y), acc);
                            acc = cfma2(xi[k], cpack(t.z, t.w), acc);
                        }
                    } else {
                        const uint16_t* h = reinterpret_cast<const uint16_t*>(in);
                        for (int k = 0; k < R; ++k) {
                            const uint32_t v = h[k];
                            const float4 t = w[k];
                            acc = cfma2(byte_pair(v, 0), cpack(t.x, t.y), acc);
                            acc = cfma2(byte_pair(v, 1), cpack(t.z, t.w), acc);
                        }
                    }
                    float ar, ai, rc, rs;
                    cunpack(acc, ar, ai);
                    rotation(incs[c0 + g] * (uint32_t) R * m, rc, rs);
                    const float bre = fmaf(ar, rc, ai * rs);          // (ar + j ai) (rc - j rs)
                    const float bim = fmaf(ai, rc, -(ar * rs));
                    if (!RUNS && p.baseband != nullptr && j >= 32 && j < 4 * ta + 32)
                        p.baseband[((int64_t) s * C + c0 + g) * p.baseband_stride + 4 * n0 + (j - 32)] = make_float2(bre, bim);
                    const float ph = atan2_approx_dev(bim, bre);
                    const float prev = __shfl_up_sync(0xffffffffu, ph, 1);
                    if (lane > 0) demod[g * FC_DEMOD + j] = fm_limit(ph, prev);
                }
            }
            __syncthreads();
            // the input stage is consumed after the last group: refill it with the tile n_stages steps ahead
            if (c0 + G >= C && tid == 0) {
                const int64_t nxt = tile + n_stages * (int64_t) gridDim.x;
                if (nxt < total_tiles) {
                    fence_proxy_async_smem();
                    issue(nxt, st);
                }
            }

            // ---- 2. half-band #1 (audio_main.c:133); work index 0 <-> 2*n0 - 10 ----
            for (int i = tid; i < gc * FC_NW; i += FC_THREADS) {
                const int g = i / FC_NW, mm = i - g * FC_NW;
                work[g * FC_WORK + mm] = halfband_from(demod + g * FC_DEMOD + 2 * mm + 2);
            }
            __syncthreads();

            // ---- 3. half-band #2 (audio_main.c:139) ----
            for (int i = tid; i < gc * FC_T; i += FC_THREADS) {
                const int g = i / FC_T, a = i - g * FC_T;
                if (a < ta)
                    p.audio[((RUNS ? run->audio_row : (int64_t) s * C) + c0 + g) * p.audio_stride + n0 + a] = halfband_from(work + g * FC_WORK + 2 * a);
            }
            // taps[] are rewritten by the next group after every thread passed the phase-1 barrier; demod[] in the
            // next phase 1, after the phase-2 barrier; work[] in the next phase 2, after the next phase-1 barrier,
            // which every phase-3 reader reaches first.
        }
    }
}

template <int RT, int G>
__global__ void __launch_bounds__(FC_THREADS) fm_channels_kernel(const FcParams p, const int tiles_per_stream,
                                                                 const int stage_bytes, const int n_stages)
{
    fm_channels_tiles<RT, G, false>(p, tiles_per_stream, stage_bytes, n_stages);
}

template <int RT, int G>
__global__ void __launch_bounds__(FC_THREADS) fm_channels_runs_kernel(const __grid_constant__ FcRunsParams p,
                                                                      const int tiles_per_stream,
                                                                      const int stage_bytes, const int n_stages)
{
    fm_channels_tiles<RT, G, true>(p, tiles_per_stream, stage_bytes, n_stages);
}

// One launch of fm_channels_kernel or fm_channels_runs_kernel at G channels per group; p.n_streams counts IQ rows or
// runs
template <class P>
int launch_fc(void (*kern)(P, int, int, int), int G, const P& p, int64_t tps, cudaStream_t stream)
{
    const int R = p.R;
    const int stage_bytes = FC_ND * 2 * R;
    const int n_stages = 2 * stage_bytes <= 120 * 1024 ? 2 : 1;      // R <= 109 double-buffers; up to R = 256 one stage
    const int smem = n_stages * stage_bytes + G * R * 16 + G * (FC_DEMOD + FC_WORK) * 4 + 16;
    if (int rc = ensure_dynamic_smem((const void*) kern, smem)) return rc;
    const int per_sm = cached_occupancy((const void*) kern, FC_THREADS, smem);
    int64_t grid = (int64_t) sm_count() * per_sm;
    const int64_t total = (int64_t) p.n_streams * tps;
    if (grid > total) grid = total;
    kern<<<(unsigned) grid, FC_THREADS, smem, stream>>>(p, (int) tps, stage_bytes, n_stages);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

// The checks the uniform and the runs calls share.  n_rows counts IQ rows (uniform) or runs: with the tiles per
// stream, returned in *tps, it bounds the launch's tile count.
int check_channel_args(const char* who, const uint8_t* iq, int64_t stream_stride_bytes, int n_rows, int64_t n_samples,
                       int R, const float* audio, int64_t audio_stride, const float* taps, int T, int64_t* tps)
{
    if (iq == nullptr || audio == nullptr) {
        set_error("%s: null IQ or audio pointer", who);
        return B200_ERR_ARG;
    }
    if (R < 1 || R > 256) {
        set_error("%s: down factor %d outside [1, 256]", who, R);
        return B200_ERR_ARG;
    }
    if (n_samples < 0 || n_samples % (4 * R) != 0 || n_samples % 8 != 0) {
        set_error("%s: n_samples %lld must be a multiple of 4*R and of 8", who, (long long) n_samples);
        return B200_ERR_ARG;
    }
    if ((taps != nullptr || T != 0) && (taps == nullptr || T < 1 || T > B200_FM_MAX_CHANNEL_TAPS)) {
        set_error("%s: %d taps: want NULL taps and 0 (boxcar) or [1, %d] device taps", who, T, B200_FM_MAX_CHANNEL_TAPS);
        return B200_ERR_ARG;
    }
    const int64_t n_audio = n_samples / (4 * R);
    if (audio_stride < n_audio) {       // overlapping rows would race
        set_error("%s: audio rows %lld floats apart for %lld samples a row", who, (long long) audio_stride,
                  (long long) n_audio);
        return B200_ERR_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(iq) & 15) != 0 || (stream_stride_bytes & 15) != 0) {
        set_error("%s: IQ pointer and stream stride must be 16-byte aligned", who);
        return B200_ERR_ALIGN;
    }
    if ((reinterpret_cast<uintptr_t>(audio) & 3) != 0 || (reinterpret_cast<uintptr_t>(taps) & 3) != 0) {
        set_error("%s: audio and taps must be 4-byte aligned", who);
        return B200_ERR_ALIGN;
    }
    *tps = (n_audio + FC_T - 1) / FC_T;
    if ((int64_t) n_rows * *tps >= (1ll << 31)) {
        set_error("%s: batch too long", who);
        return B200_ERR_ARG;
    }
    return B200_OK;
}

}  // namespace

int launch_fm_channels_runs(const uint8_t* iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                            const b200_fm_channel_run* runs, int n_runs, float* audio, int64_t audio_stride,
                            int64_t n_audio_rows, const float* taps, int T, cudaStream_t stream)
{
    int64_t tps;
    if (int rc = check_channel_args("fm channels runs", iq, stream_stride_bytes, n_runs, n_samples, R, audio,
                                    audio_stride, taps, T, &tps))
        return rc;
    if (runs == nullptr || n_streams < 1 || n_runs < 1 || n_runs > B200_FM_MAX_RUNS || n_audio_rows < 1) {
        set_error("fm channels runs: %d runs (table %p) over %d IQ rows, %lld audio rows; want [1, %d] runs, at least one "
                  "row of each", n_runs, (const void*) runs, n_streams, (long long) n_audio_rows, B200_FM_MAX_RUNS);
        return B200_ERR_ARG;
    }
    int max_c = 0;
    for (int k = 0; k < n_runs; ++k) {
        const b200_fm_channel_run& r = runs[k];
        if (r.stream < 0 || r.stream >= n_streams || r.n_channels < 1 || r.n_channels > B200_FM_MAX_CHANNELS ||
            r.first_sample < 0 || r.first_sample % (4 * R) != 0 || r.audio_row < 0 ||
            r.audio_row > n_audio_rows - r.n_channels) {
            set_error("fm channels runs: run %d (row %d of %d, %d channels, first sample %lld, audio row %lld of %lld)",
                      k, r.stream, n_streams, r.n_channels, (long long) r.first_sample, (long long) r.audio_row,
                      (long long) n_audio_rows);
            return B200_ERR_ARG;
        }
        // two runs writing the same audio row would race
        for (int i = 0; i < k; ++i)
            if (r.audio_row < runs[i].audio_row + runs[i].n_channels && runs[i].audio_row < r.audio_row + r.n_channels) {
                set_error("fm channels runs: the audio rows of runs %d and %d overlap", i, k);
                return B200_ERR_ARG;
            }
        if (r.n_channels > max_c) max_c = r.n_channels;
    }
    if (n_samples == 0) return B200_OK;
    FcRunsParams p;
    memset(&p, 0, sizeof(p));
    p.iq = iq;
    p.stream_stride_bytes = stream_stride_bytes;
    p.n_streams = n_runs;
    p.n_samples = n_samples;
    p.R = R;
    p.audio = audio;
    p.audio_stride = audio_stride;
    for (int k = 0; k < n_runs; ++k) {
        FcRun& r = p.runs[k];
        r.stream = runs[k].stream;
        r.n_channels = runs[k].n_channels;
        r.first_dec = (uint32_t) (runs[k].first_sample / R);
        r.audio_row = runs[k].audio_row;
        memcpy(r.phase_inc, runs[k].phase_inc, sizeof(r.phase_inc));
    }
    if (taps != nullptr) return launch_fm_channels_fir_runs(p, tps, taps, T, max_c, stream);
    if (R == 10) return launch_fc(fm_channels_runs_kernel<10, 8>, 8, p, tps, stream);
    return launch_fc(fm_channels_runs_kernel<0, 4>, 4, p, tps, stream);
}

int launch_fm_channels(const uint8_t* iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                       int64_t first_sample, const uint32_t* phase_inc, int n_channels, float* audio,
                       int64_t audio_stride, float* baseband, int64_t baseband_stride, const float* taps, int T,
                       cudaStream_t stream)
{
    int64_t tps;
    if (int rc = check_channel_args("fm channels", iq, stream_stride_bytes, n_streams, n_samples, R, audio,
                                    audio_stride, taps, T, &tps))
        return rc;
    if (n_streams < 0 || phase_inc == nullptr) {
        set_error("fm channels: null phase increments or negative stream count");
        return B200_ERR_ARG;
    }
    if (n_channels < 1 || n_channels > B200_FM_MAX_CHANNELS) {
        set_error("fm channels: n_channels %d outside [1, %d]", n_channels, B200_FM_MAX_CHANNELS);
        return B200_ERR_ARG;
    }
    if (first_sample < 0 || first_sample % (4 * R) != 0) {
        set_error("fm channels: first_sample %lld must be a non-negative multiple of 4*R", (long long) first_sample);
        return B200_ERR_ARG;
    }
    if (baseband != nullptr && baseband_stride < n_samples / R) {      // overlapping rows would race
        set_error("fm channels: baseband rows %lld samples apart for %lld samples a row", (long long) baseband_stride,
                  (long long) (n_samples / R));
        return B200_ERR_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(phase_inc) & 3) != 0 || (reinterpret_cast<uintptr_t>(baseband) & 7) != 0) {
        set_error("fm channels: phase increments must be 4-byte aligned, baseband 8-byte aligned");
        return B200_ERR_ALIGN;
    }
    if (n_streams == 0 || n_samples == 0) return B200_OK;
    FcParams p;
    p.iq = iq;
    p.stream_stride_bytes = stream_stride_bytes;
    p.n_streams = n_streams;
    p.n_samples = n_samples;
    p.R = R;
    p.first_sample = first_sample;
    p.phase_inc = phase_inc;
    p.n_channels = n_channels;
    p.audio = audio;
    p.audio_stride = audio_stride;
    p.baseband = reinterpret_cast<float2*>(baseband);
    p.baseband_stride = baseband_stride;
    if (taps != nullptr) return launch_fm_channels_fir(p, tps, taps, T, stream);
    // channels per group at R = 10: 8 measured fastest at every channel count (DESIGN.md 4.3a)
    if (R == 10) return launch_fc(fm_channels_kernel<10, 8>, 8, p, tps, stream);
    return launch_fc(fm_channels_kernel<0, 4>, 4, p, tps, stream);
}

}  // namespace b200

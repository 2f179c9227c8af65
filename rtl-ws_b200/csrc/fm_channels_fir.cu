// fm_channels_fir.cu -- FM channels with a T-tap FIR low-pass in place of the boxcar (sm_100a).
//
// Same chain as fm_channels.cu (include/b200sdr.h), but the decimating filter in front of the demodulator is
//   b[m] = sum_{k<T} h[k] y[mR + R - T + k],   y[n] = x[n] exp(-j 2 pi phi(n) / 2^32)
// with real taps h: its last tap sits on the last sample of the boxcar's window, so T = R, h = 1 is the boxcar.
// Write L = T - R (any sign).  phi(mR + d) = phi(mR) + phi(d) mod 2^32 holds for negative d too (uint32 two's
// complement), so
//   b[m] = exp(-j phi(mR)) * sum_{k<T} x[mR - L + k] w[k],   w[k] = h[k] exp(-j 2 pi phi(k - L) / 2^32):
// one complex T-tap filter per channel, then the same exact-integer rotation per decimated sample as the boxcar.
//
// Geometry: the boxcar kernel's tile (280 decimated samples, 9 warps, one 31-output discriminator chunk per warp)
// and TMA ring.  A stage holds 280 R + L input samples; the bulk copy starts at the 8-sample boundary at or below
// the first one a tile needs, off = (-L) mod 8 samples ahead of it, so lane j's window starts at stage sample
// j R + off.  The MAC reads byte pairs straight from the stage (2 bytes per sample: the stage of R = 256, T = 1024
// is 142 KB, its floats would not fit), unpacks each once and applies it to the G channels of the group:
// G accumulators per lane, taps [T][G] in shared memory, read as broadcasts.  G comes from the shared-memory budget
// and the channel count (launcher).  Phases 2 and 3 (the half-bands) are the boxcar kernel's.
#include <math.h>
#include <string.h>

#include "b200_common.cuh"
#include "fm_channels.cuh"
#include "fm_kernels.cuh"

namespace b200 {

namespace {

constexpr int FIR_MAX_G = 8;                       // channels per group (accumulators per lane)
constexpr int FIR_SMEM_LIMIT = 227 * 1024;         // dynamic shared memory a B200 CTA may opt into

struct FirParams {
    FcParams c;
    const float* taps;              // [T], shared by every channel and stream
    int T;
    int L;                          // T - R
    int off;                        // (-L) mod 8: where lane 0's window starts in a stage
};

// the runs form: c.n_streams counts runs (FcRunsParams)
struct FirRunsParams : FirParams {
    FcRun runs[B200_FM_MAX_RUNS];
};

// MAC over T taps for NG channels of the group, then rotation, discriminator and limiter -> demod[g][j]
// bb (nullable): this tile's baseband column 0 of channel 0 of the group, rows bb_stride complex samples apart
template <int NG>
__device__ __forceinline__ void fir_group(const uint16_t* in, const float4* taps, int T, int G, int R,
                                          const uint32_t* incs, uint32_t m, int j, int lane, float2* bb,
                                          int64_t bb_stride, int ta, float* demod)
{
    c64 acc[NG];
#pragma unroll
    for (int g = 0; g < NG; ++g) acc[g] = cpack(0.0f, 0.0f);
#pragma unroll 4
    for (int k = 0; k < T; ++k) {
        const uint32_t v = in[k];
        const c64 xr = byte_pair(v, 0);
        const c64 xi = byte_pair(v, 1);
        const float4* t = taps + k * G;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            const float4 w = t[g];
            acc[g] = cfma2(xr, cpack(w.x, w.y), acc[g]);
            acc[g] = cfma2(xi, cpack(w.z, w.w), acc[g]);
        }
    }
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        float ar, ai, rc, rs;
        cunpack(acc[g], ar, ai);
        rotation(incs[g] * (uint32_t) R * m, rc, rs);
        const float bre = fmaf(ar, rc, ai * rs);          // (ar + j ai) (rc - j rs)
        const float bim = fmaf(ai, rc, -(ar * rs));
        if (bb != nullptr && j >= 32 && j < 4 * ta + 32) bb[g * bb_stride + (j - 32)] = make_float2(bre, bim);
        const float ph = atan2_approx_dev(bim, bre);
        const float prev = __shfl_up_sync(0xffffffffu, ph, 1);
        if (lane > 0) demod[g * FC_DEMOD + j] = fm_limit(ph, prev);
    }
}

// the tile loop of both forms, as fm_channels_tiles in fm_channels.cu
template <bool RUNS, class P>
__device__ __forceinline__ void fm_channels_fir_tiles(const P& p, const int tiles_per_stream, const int stage_bytes,
                                                      const int n_stages, const int G)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int R = p.c.R;
    const int T = p.T;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    uint8_t* ring = smem;
    float4* taps = reinterpret_cast<float4*>(smem + n_stages * stage_bytes);   // [T][G]: (w.re, w.im, -w.im, w.re)
    float* demod = reinterpret_cast<float*>(taps + T * G);                        // [G][FC_DEMOD]
    float* work = demod + G * FC_DEMOD;                                           // [G][FC_WORK]
    uint64_t* bars = reinterpret_cast<uint64_t*>(work + G * FC_WORK);

    const int C_all = p.c.n_channels;
    const int64_t n_audio = p.c.n_samples / (4 * R);
    const int64_t total_tiles = (int64_t) p.c.n_streams * tiles_per_stream;
    const uint32_t first_dec_all = (uint32_t) (p.c.first_sample / R);      // mod 2^32, like every phase below

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
        // samples from (4 n0 - 32) R - L - off (a multiple of 8: (4 n0 - 32) R is one because n0 is a multiple of 62,
        // and L + off is one by the choice of off) up to 4 (n0 + ta) R, a multiple of 8 as in fm_channels.cu
        const int64_t first = (4 * n0 - 32) * (int64_t) R - p.L - p.off;
        const uint32_t bytes = (uint32_t) (2 * ((4 * (n0 + ta)) * (int64_t) R - first));
        const uint8_t* src = p.c.iq + (int64_t) s * p.c.stream_stride_bytes + 2 * first;
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
        const uint32_t* incs = RUNS ? run->phase_inc : p.c.phase_inc + (int64_t) s * C;

        mbar_wait(&bars[st], (it / (uint32_t) n_stages) & 1);
        // lane j's window: input samples (4 n0 - 32 + j) R - L + k, k < T
        const uint16_t* in = reinterpret_cast<const uint16_t*>(ring + st * stage_bytes) + j * R + p.off;

        for (int c0 = 0; c0 < C; c0 += G) {
            const int gc = (C - c0) < G ? (C - c0) : G;
            // ---- 0. taps of the group: h[k] exp(-j 2 pi phi(k - L) / 2^32) ----
            for (int i = tid; i < gc * T; i += FC_THREADS) {
                const int g = i / T, k = i - g * T;
                const uint32_t phi = incs[c0 + g] * (uint32_t) (k - p.L);
                float sn, cs;
                sincospif((float) (int32_t) phi * 4.65661287307739258e-10f, &sn, &cs);     // 2^-31: [-1, 1)
                const float h = p.taps[k];
                taps[k * G + g] = make_float4(h * cs, -(h * sn), h * sn, h * cs);
            }
            __syncthreads();

            // ---- 1. mix + FIR, rotation, discriminator ----
            float2* bb = !RUNS && p.c.baseband != nullptr
                             ? p.c.baseband + ((int64_t) s * C + c0) * p.c.baseband_stride + 4 * n0 : nullptr;
            const int64_t bs = p.c.baseband_stride;
            switch (gc) {
                case 1: fir_group<1>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 2: fir_group<2>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 3: fir_group<3>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 4: fir_group<4>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 5: fir_group<5>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 6: fir_group<6>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                case 7: fir_group<7>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
                default: fir_group<8>(in, taps, T, G, R, incs + c0, m, j, lane, bb, bs, ta, demod); break;
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
                    p.c.audio[((RUNS ? run->audio_row : (int64_t) s * C) + c0 + g) * p.c.audio_stride + n0 + a] = halfband_from(work + g * FC_WORK + 2 * a);
            }
            // taps[], demod[] and work[] are reused under the same barriers as in fm_channels.cu
        }
    }
}

__global__ void __launch_bounds__(FC_THREADS) fm_channels_fir_kernel(const FirParams p, const int tiles_per_stream,
                                                                     const int stage_bytes, const int n_stages,
                                                                     const int G)
{
    fm_channels_fir_tiles<false>(p, tiles_per_stream, stage_bytes, n_stages, G);
}

// three CTAs per SM, as the uniform kernel (72 registers): unbounded, the per-run values take this one to 81, which
// leaves room for only two 288-thread CTAs
__global__ void __launch_bounds__(FC_THREADS, 3) fm_channels_fir_runs_kernel(const __grid_constant__ FirRunsParams p,
                                                                          const int tiles_per_stream,
                                                                          const int stage_bytes, const int n_stages,
                                                                          const int G)
{
    fm_channels_fir_tiles<true>(p, tiles_per_stream, stage_bytes, n_stages, G);
}

constexpr int fir_stage_bytes(int R, int T)
{
    const int L = T - R;
    return 2 * (FC_ND * R + L + ((-L) & 7));
}

constexpr int fir_smem_bytes(int stage_bytes, int n_stages, int T, int G)
{
    return n_stages * stage_bytes + T * G * 16 + G * (FC_DEMOD + FC_WORK) * 4 + 16;
}

// One channel per group fits at every R and T: the largest stage (R = 256, T = B200_FM_MAX_CHANNEL_TAPS, 142 KB) is
// single-buffered, and two stages take at most 120 KB
static_assert(fir_smem_bytes(fir_stage_bytes(256, B200_FM_MAX_CHANNEL_TAPS), 1, B200_FM_MAX_CHANNEL_TAPS, 1) <=
                  FIR_SMEM_LIMIT, "the largest FIR channel stage does not fit in shared memory");

// Channels per group for C channels: the fewest groups the shared-memory budget allows (at most FIR_MAX_G
// channels each), then the channels spread evenly over them
int fir_group_size(int stage_bytes, int n_stages, int T, int C)
{
    int gmax = C < FIR_MAX_G ? C : FIR_MAX_G;
    while (gmax > 1 && fir_smem_bytes(stage_bytes, n_stages, T, gmax) > FIR_SMEM_LIMIT) --gmax;
    const int groups = (C + gmax - 1) / gmax;
    return (C + groups - 1) / groups;
}

// One launch of fm_channels_fir_kernel or fm_channels_fir_runs_kernel: fills the filter fields of p (p.c is set;
// p.c.n_streams counts IQ rows or runs), G from the largest channel count
template <class P>
int launch_fir(void (*kern)(P, int, int, int, int), P& p, int64_t tps, const float* taps, int T, int max_channels,
               cudaStream_t stream)
{
    const int R = p.c.R;
    const int stage_bytes = fir_stage_bytes(R, T);
    const int n_stages = 2 * stage_bytes <= 120 * 1024 ? 2 : 1;       // as fm_channels.cu
    const int G = fir_group_size(stage_bytes, n_stages, T, max_channels);
    p.taps = taps;
    p.T = T;
    p.L = T - R;
    p.off = (R - T) & 7;
    const int smem = fir_smem_bytes(stage_bytes, n_stages, T, G);
    if (int rc = ensure_dynamic_smem((const void*) kern, smem)) return rc;
    const int per_sm = cached_occupancy((const void*) kern, FC_THREADS, smem);
    int64_t grid = (int64_t) sm_count() * per_sm;
    const int64_t total = (int64_t) p.c.n_streams * tps;
    if (grid > total) grid = total;
    kern<<<(unsigned) grid, FC_THREADS, smem, stream>>>(p, (int) tps, stage_bytes, n_stages, G);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace

int launch_fm_channels_fir(const FcParams& c, int64_t tps, const float* taps, int T, cudaStream_t stream)
{
    FirParams p;
    p.c = c;
    return launch_fir(fm_channels_fir_kernel, p, tps, taps, T, c.n_channels, stream);
}

// a run's audio does not depend on G (each channel's MAC, rotation and demodulator are the same whatever group it is
// computed in)
int launch_fm_channels_fir_runs(const FcRunsParams& runs, int64_t tps, const float* taps, int T, int max_channels,
                                cudaStream_t stream)
{
    FirRunsParams p;
    p.c = runs;
    memcpy(p.runs, runs.runs, sizeof(p.runs));
    return launch_fir(fm_channels_fir_runs_kernel, p, tps, taps, T, max_channels, stream);
}

int fm_channels_fir_history_samples(int R, int T)
{
    if (R < 1 || R > 256 || T < 1 || T > B200_FM_MAX_CHANNEL_TAPS) return B200_ERR_ARG;
    const int h = 32 * R + (T > R ? T - R : 0);
    return (h + 7) / 8 * 8;
}

int IqRows::set_channel_filter(const char* who, const float* h_taps, int count, cudaStream_t stream)
{
    if (count < 0 || count > B200_FM_MAX_CHANNEL_TAPS || (count > 0 && h_taps == nullptr)) {
        set_error("%s: bad arguments (%d taps)", who, count);
        return B200_ERR_ARG;
    }
    const int h = count > 0 ? fm_channels_fir_history_samples(R, count) : fm_history_samples(R);
    // the carry copies within a row: a history longer than the batch would overlap its own source
    if (h > max_batch) {
        set_error("%s: its history of %d samples is longer than the batch (%lld)", who, h, (long long) max_batch);
        return B200_ERR_ARG;
    }
    float* taps = nullptr;
    cudaError_t e = cudaSuccess;
    if (count > 0) {
        e = cudaMalloc((void**) &taps, sizeof(float) * (size_t) count);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(taps, h_taps, sizeof(float) * (size_t) count, cudaMemcpyHostToDevice, stream);
    }
    IqRows fresh{R, n_rows, max_batch};     // rows with the new history; at position 0 nothing in the old ones is kept
    int rc = B200_OK;
    if (e == cudaSuccess && h != hist)
        rc = fresh.alloc(h, stream);        // also waits for the taps
    else if (e == cudaSuccess)
        e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        set_error("%s: %s", who, cudaGetErrorString(e));
        rc = B200_ERR_CUDA;
    }
    if (rc != B200_OK) {
        cudaFree(taps);
        fresh.free();
        return rc;
    }
    if (fresh.d_base != nullptr) {
        cudaFree(d_base);
        d_base = fresh.d_base;
        pitch = fresh.pitch;
        hist = h;
    }
    cudaFree(d_taps);
    d_taps = taps;
    n_taps = count;
    return B200_OK;
}

// Kaiser-windowed sinc (host): I0 by its power series, which converges for every beta used here (< 120)
static double bessel_i0(double x)
{
    double sum = 1.0, term = 1.0;
    const double q = 0.25 * x * x;
    for (int k = 1; k < 500; ++k) {
        term *= q / ((double) k * (double) k);
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

int fm_channel_filter_design(int R, int T, double cutoff_hz, double atten_db, double fs, float* h)
{
    // !(a < b) also refuses NaN
    if (h == nullptr || R < 1 || R > 256 || T < 1 || T > B200_FM_MAX_CHANNEL_TAPS || !(fs > 0.0) || !isfinite(fs) ||
        !(cutoff_hz > 0.0) || !(cutoff_hz < 0.5 * fs) || !(atten_db >= 0.0) || !isfinite(atten_db)) {
        set_error("fm channel filter design: R %d, %d taps, cutoff %g Hz, attenuation %g dB, rate %g Hz", R, T,
                  cutoff_hz, atten_db, fs);
        return B200_ERR_ARG;
    }
    const double A = atten_db;
    const double beta = A > 50.0 ? 0.1102 * (A - 8.7) : A >= 21.0 ? 0.5842 * pow(A - 21.0, 0.4) + 0.07886 * (A - 21.0) : 0.0;
    const double fc = cutoff_hz / fs;                        // cycles per sample; the -6 dB point of the windowed sinc
    const double mid = 0.5 * (T - 1);
    const double pi = 3.14159265358979323846;
    const double i0b = bessel_i0(beta);
    double v[B200_FM_MAX_CHANNEL_TAPS];
    double sum = 0.0;
    for (int k = 0; k < T; ++k) {
        const double t = k - mid;
        const double sinc = t == 0.0 ? 2.0 * fc : sin(2.0 * pi * fc * t) / (pi * t);
        const double r = T > 1 ? (k - mid) / mid : 0.0;
        const double w = bessel_i0(beta * sqrt(fmax(0.0, 1.0 - r * r))) / i0b;
        v[k] = sinc * w;
        sum += v[k];
    }
    if (!(fabs(sum) > 0.0)) {
        set_error("fm channel filter design: the taps sum to zero");
        return B200_ERR_ARG;
    }
    // the boxcar's DC gain R, so the baseband keeps the scale the demodulator was checked at
    for (int k = 0; k < T; ++k) h[k] = (float) (v[k] * (double) R / sum);
    return B200_OK;
}

}  // namespace b200

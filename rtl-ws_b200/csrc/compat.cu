// compat.cu -- the reference's own DSP interface, symbol for symbol, over the CUDA kernels
// (declared in include/rtlws_compat.h).  An unmodified cbb_main.c / audio_main.c / main.c
// links against these instead of spectrum.o, rf_decimator.o and resample.o.
//
//   spectrum.h:9-17      spectrum_alloc / spectrum_add_{cmplx_u8,cmplx_s32,real_f32} / spectrum_free
//   rf_decimator.h:11-21 rf_decimator_{alloc,add_callback,set_parameters,decimate_cmplx_u8,
//                        remove_callbacks,free}
//   resample.h:14-17     cic_decimate / halfband_decimate
//
// These calls are synchronous and small (2 KB in / 8 KB out for a spectrum), so they are
// bound by launch and PCIe latency, not bandwidth: they exist for drop-in correctness.
// Throughput goes through the batched entry points of b200sdr.h.
// Error convention follows the reference: 0 ok, -1 size/parameter mismatch, -2 internal
// failure (which here includes any CUDA error; it is logged to stderr like log.h's ERROR).
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/rtlws_compat.h"
#include "b200_common.cuh"
#include "fm_kernels.cuh"

using namespace b200;

namespace {

#define COMPAT_LOG(...)                                 \
    do {                                                \
        fprintf(stderr, "libb200sdr %s:%d [E] ", __FILE__, __LINE__); \
        fprintf(stderr, __VA_ARGS__);                   \
        fprintf(stderr, "\n");                          \
    } while (0)

// ---- small kernels used only by the compat calls ------------------------------------------

// spectrum.c:23-34 accumulate-into-caller semantics: ps[i] += P[i] except at the DC
// position, which adds its (already updated) left neighbour.
__global__ void accumulate_ps_kernel(double* ps, const float* pw, int N)
{
    const int half = N / 2;
    for (int i = threadIdx.x; i < N; i += blockDim.x)
        if (i != half) ps[i] += (double) pw[i];
    __syncthreads();
    if (threadIdx.x == 0) ps[half] += ps[half - 1];
}

// resample.c:21-40: boxcar sums of R samples minus 128*R; out[0] additionally carries the
// caller's (integrator_prev_out - comb_prev_in), which is zero for any state the
// reference itself can produce.  Per-block partial sums feed the integrator write-back.
__global__ void cic_kernel(const uint16_t* __restrict__ src, int2* __restrict__ dst, int dst_len, int R, int adj_re,
                           int adj_im, unsigned int* __restrict__ totals)
{
    unsigned int tre = 0, tim = 0;
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < dst_len; m += gridDim.x * blockDim.x) {
        const uint16_t* s = src + (size_t) m * R;
        unsigned int ure = 0, uim = 0;
        for (int k = 0; k < R; ++k) {
            const unsigned int v = s[k];
            ure += v & 0xffu;
            uim += v >> 8;
        }
        const unsigned int bre = ure - 128u * (unsigned int) R;
        const unsigned int bim = uim - 128u * (unsigned int) R;
        tre += bre;
        tim += bim;
        dst[m] = make_int2((int) (bre + (m == 0 ? (unsigned int) adj_re : 0u)),
                           (int) (bim + (m == 0 ? (unsigned int) adj_im : 0u)));
    }
    for (int o = 16; o > 0; o >>= 1) {
        tre += __shfl_down_sync(0xffffffffu, tre, o);
        tim += __shfl_down_sync(0xffffffffu, tim, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&totals[0], tre);
        atomicAdd(&totals[1], tim);
    }
}

// resample.c:47-64 over ext = [10 delay floats | input]
__global__ void halfband_kernel(const float* __restrict__ ext, float* __restrict__ out, int output_len)
{
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < output_len; n += gridDim.x * blockDim.x) {
        const float* x = ext + 2 * n + 10;      // x[-k] = input[2n - k]
        out[n] = halfband_taps(x[0], x[-2], x[-4], x[-5], x[-6], x[-8], x[-10]);
    }
}

// grow-only device + pinned scratch, one per handle or per thread
struct Scratch {
    void* d = nullptr;
    void* h = nullptr;
    size_t bytes = 0;
    bool reserve(size_t need)
    {
        if (need <= bytes) return true;
        if (d) cudaFree(d);
        if (h) cudaFreeHost(h);
        d = h = nullptr;
        bytes = 0;
        if (cudaMalloc(&d, need) != cudaSuccess) return false;
        if (cudaHostAlloc(&h, need, cudaHostAllocDefault) != cudaSuccess) return false;
        bytes = need;
        return true;
    }
    void release()
    {
        if (d) cudaFree(d);
        if (h) cudaFreeHost(h);
        d = h = nullptr;
        bytes = 0;
    }
};

thread_local Scratch t_scratch;

}  // namespace

// =============================== spectrum.h ==========================================

struct spectrum {
    int N;
    b200_spectrum_plan* plan;
    Scratch buf;        // device: [input 8N | power 4N | ps 8N], pinned mirror of the same
    cudaStream_t stream;
};

extern "C" {

struct spectrum* spectrum_alloc(int N)
{
    // spectrum.c:37-45 plans with FFTW for any N; this build transforms powers of two
    struct spectrum* s = new spectrum();
    s->N = N;
    s->plan = b200_spectrum_plan_create(N, N, 1, N, B200_WINDOW_RECT, 0);
    s->stream = nullptr;
    if (s->plan == nullptr || !s->buf.reserve((size_t) N * 20) ||
        cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) {
        COMPAT_LOG("spectrum_alloc(%d) failed: %s", N, b200_last_error());
        if (s->plan) b200_spectrum_plan_destroy(s->plan);
        s->buf.release();
        delete s;
        return nullptr;
    }
    return s;
}

static int spectrum_add_any(struct spectrum* s, const void* src, size_t in_bytes, double* power_spectrum, int len,
                            int kind)
{
    if (s == nullptr || len != s->N)      // spectrum.c:51-52
        return -1;
    const int N = s->N;
    uint8_t* d_in = (uint8_t*) s->buf.d;
    float* d_pw = (float*) (d_in + (size_t) N * 8);
    double* d_ps = (double*) (d_in + (size_t) N * 12);
    uint8_t* h_in = (uint8_t*) s->buf.h;
    double* h_ps = (double*) (h_in + (size_t) N * 12);
    memcpy(h_in, src, in_bytes);
    memcpy(h_ps, power_spectrum, sizeof(double) * (size_t) N);
    bool ok = cudaMemcpyAsync(d_in, h_in, in_bytes, cudaMemcpyHostToDevice, s->stream) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(d_ps, h_ps, sizeof(double) * (size_t) N, cudaMemcpyHostToDevice, s->stream) == cudaSuccess;
    int rc = 0;
    if (ok) {
        if (kind == 0)
            rc = b200_spectrum_exec(s->plan, d_in, 0, 1, 1, nullptr, d_pw, nullptr, s->stream);
        else if (kind == 1)
            rc = b200_spectrum_exec_cs32(s->plan, (const int32_t*) d_in, 0, 1, 1, nullptr, d_pw, nullptr, s->stream);
        else
            rc = b200_spectrum_exec_rf32(s->plan, (const float*) d_in, 0, 1, 1, nullptr, d_pw, nullptr, s->stream);
    }
    if (ok && rc == 0) {
        accumulate_ps_kernel<<<1, 1024, 0, s->stream>>>(d_ps, d_pw, N);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        ok = cudaGetLastError() == cudaSuccess;
        ok = ok && cudaMemcpyAsync(h_ps, d_ps, sizeof(double) * (size_t) N, cudaMemcpyDeviceToHost, s->stream) == cudaSuccess;
        ok = ok && cudaStreamSynchronize(s->stream) == cudaSuccess;
    }
    if (!ok || rc != 0) {
        COMPAT_LOG("spectrum_add: %s", rc ? b200_last_error() : cudaGetErrorString(cudaGetLastError()));
        return -2;
    }
    memcpy(power_spectrum, h_ps, sizeof(double) * (size_t) N);
    return 0;
}

int spectrum_add_cmplx_u8(struct spectrum* s, const cmplx_u8* src, double* power_spectrum, int len)
{
    return spectrum_add_any(s, src, (size_t) (len > 0 ? len : 0) * 2, power_spectrum, len, 0);
}

int spectrum_add_cmplx_s32(struct spectrum* s, const cmplx_s32* src, double* power_spectrum, int len)
{
    return spectrum_add_any(s, src, (size_t) (len > 0 ? len : 0) * 8, power_spectrum, len, 1);
}

int spectrum_add_real_f32(struct spectrum* s, const float* src, double* power_spectrum, int len)
{
    return spectrum_add_any(s, src, (size_t) (len > 0 ? len : 0) * 4, power_spectrum, len, 2);
}

void spectrum_free(struct spectrum* s)
{
    if (s == nullptr) return;
    if (s->stream) cudaStreamDestroy(s->stream);
    b200_spectrum_plan_destroy(s->plan);
    s->buf.release();
    delete s;
}

// =============================== resample.h ==========================================

int cic_decimate(int R, const cmplx_u8* src, int src_len, cmplx_s32* dst, int dst_len, struct cic_delay_line* delay)
{
    if (R < 1 || dst_len * R != src_len)          // resample.c:18-19
        return -1;
    if (dst_len == 0) return 0;
    Scratch& sc = t_scratch;
    const size_t in_bytes = (size_t) src_len * 2;
    const size_t out_bytes = (size_t) dst_len * 8;
    const size_t in_pad = (in_bytes + 255) & ~(size_t) 255;
    if (!sc.reserve(in_pad + out_bytes + 256)) {
        COMPAT_LOG("cic_decimate: scratch allocation failed");
        return -2;
    }
    uint8_t* d_in = (uint8_t*) sc.d;
    int2* d_out = (int2*) (d_in + in_pad);
    unsigned int* d_tot = (unsigned int*) (d_in + in_pad + out_bytes);
    unsigned int h_tot[2] = {0, 0};
    const unsigned int integ_re = (unsigned int) delay->integrator_prev_out.p.re;
    const unsigned int integ_im = (unsigned int) delay->integrator_prev_out.p.im;
    const unsigned int comb_re = (unsigned int) delay->comb_prev_in.p.re;
    const unsigned int comb_im = (unsigned int) delay->comb_prev_in.p.im;
    bool ok = cudaMemcpy(d_in, src, in_bytes, cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemset(d_tot, 0, 8) == cudaSuccess;
    if (ok) {
        int blocks = (dst_len + 255) / 256;
        if (blocks > 1184) blocks = 1184;
        cic_kernel<<<blocks, 256>>>((const uint16_t*) d_in, d_out, dst_len, R, (int) (integ_re - comb_re),
                                    (int) (integ_im - comb_im), d_tot);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        ok = cudaGetLastError() == cudaSuccess;
    }
    ok = ok && cudaMemcpy(dst, d_out, out_bytes, cudaMemcpyDeviceToHost) == cudaSuccess;
    ok = ok && cudaMemcpy(h_tot, d_tot, 8, cudaMemcpyDeviceToHost) == cudaSuccess;
    if (!ok) {
        COMPAT_LOG("cic_decimate: %s", cudaGetErrorString(cudaGetLastError()));
        return -2;
    }
    // resample.c:42-43: the integrator is the running sum (mod 2^32); the comb input equals it
    // after a whole number of output samples
    delay->integrator_prev_out.p.re = (int32_t) (integ_re + h_tot[0]);
    delay->integrator_prev_out.p.im = (int32_t) (integ_im + h_tot[1]);
    delay->comb_prev_in = delay->integrator_prev_out;
    return 0;
}

void halfband_decimate(const float* input, float* output, int output_len, float* delay)
{
    if (output_len <= 0) return;
    Scratch& sc = t_scratch;
    const size_t ext_bytes = ((size_t) 2 * output_len + 10) * 4;
    const size_t ext_pad = (ext_bytes + 255) & ~(size_t) 255;
    if (!sc.reserve(ext_pad + (size_t) output_len * 4)) {
        COMPAT_LOG("halfband_decimate: scratch allocation failed");
        return;
    }
    float* d_ext = (float*) sc.d;
    float* d_out = (float*) ((uint8_t*) sc.d + ext_pad);
    bool ok = cudaMemcpy(d_ext, delay, 10 * 4, cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && cudaMemcpy(d_ext + 10, input, (size_t) 2 * output_len * 4, cudaMemcpyHostToDevice) == cudaSuccess;
    if (ok) {
        int blocks = (output_len + 255) / 256;
        if (blocks > 1184) blocks = 1184;
        halfband_kernel<<<blocks, 256>>>(d_ext, d_out, output_len);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        ok = cudaGetLastError() == cudaSuccess;
    }
    ok = ok && cudaMemcpy(output, d_out, (size_t) output_len * 4, cudaMemcpyDeviceToHost) == cudaSuccess;
    if (!ok) {
        COMPAT_LOG("halfband_decimate: %s", cudaGetErrorString(cudaGetLastError()));
        return;
    }
    // resample.c:66: the delay line becomes the last HALF_BAND_N - 1 inputs (a copy, no arithmetic).
    // Shorter inputs keep the newest of the old delay line in front, which is what "the last
    // ten samples seen" means; the reference reads out of bounds there.
    if (2 * output_len >= HALF_BAND_N - 1) {
        memcpy(delay, input + 2 * output_len - (HALF_BAND_N - 1), (HALF_BAND_N - 1) * sizeof(float));
    } else {
        const int n = 2 * output_len;
        memmove(delay, delay + n, (size_t) (HALF_BAND_N - 1 - n) * sizeof(float));
        memcpy(delay + (HALF_BAND_N - 1 - n), input, (size_t) n * sizeof(float));
    }
}

}  // extern "C"

// =============================== rf_decimator.h ======================================

struct rf_decimator {
    pthread_mutex_t mutex;
    std::vector<rf_decimator_callback> callbacks;
    double sample_rate;
    int down_factor;
    cmplx_u8* input_signal;        // pinned, input_signal_len samples
    int input_signal_len;
    int surplus;
    cmplx_s32* resampled_signal;   // pinned, resampled_signal_len samples
    int resampled_signal_len;
    uint8_t* d_in;
    int2* d_out;
    unsigned int* d_tot;
    cudaStream_t stream;
    struct cic_delay_line delay;
};

extern "C" {

struct rf_decimator* rf_decimator_alloc()
{
    struct rf_decimator* d = new rf_decimator();
    pthread_mutex_init(&d->mutex, NULL);
    d->sample_rate = 0;
    d->down_factor = 0;
    d->input_signal = nullptr;
    d->input_signal_len = 0;
    d->surplus = 0;
    d->resampled_signal = nullptr;
    d->resampled_signal_len = 0;
    d->d_in = nullptr;
    d->d_out = nullptr;
    d->d_tot = nullptr;
    d->stream = nullptr;
    memset(&d->delay, 0, sizeof(d->delay));
    return d;
}

void rf_decimator_add_callback(struct rf_decimator* d, rf_decimator_callback callback)
{
    pthread_mutex_lock(&d->mutex);
    d->callbacks.push_back(callback);
    pthread_mutex_unlock(&d->mutex);
}

static void rf_release_buffers(struct rf_decimator* d)
{
    if (d->input_signal) cudaFreeHost(d->input_signal);
    if (d->resampled_signal) cudaFreeHost(d->resampled_signal);
    if (d->d_in) cudaFree(d->d_in);
    if (d->d_out) cudaFree(d->d_out);
    if (d->d_tot) cudaFree(d->d_tot);
    d->input_signal = nullptr;
    d->resampled_signal = nullptr;
    d->d_in = nullptr;
    d->d_out = nullptr;
    d->d_tot = nullptr;
}

int rf_decimator_set_parameters(struct rf_decimator* d, double sample_rate, int down_factor)
{
    int r = -1;
    pthread_mutex_lock(&d->mutex);
    if (sample_rate > 0 && down_factor > 0) {                  // rf_decimator.c:58
        r = 0;
        if (fabs(d->sample_rate - sample_rate) > 0.0001 || d->down_factor != down_factor) {   // :60, EPSILON :11
            const int out_len = (int) ((sample_rate / down_factor) * 100 / 1000);   // :65, INTERNAL_BUF_LEN_MS :10
            const int in_len = out_len * down_factor;                                // :66
            // carry the bytes already buffered across the reallocation, as realloc() does at :69;
            // the reference then forgets them by zeroing surplus (:71), and so does this
            rf_release_buffers(d);
            bool ok = true;
            if (d->stream == nullptr) ok = cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) == cudaSuccess;
            ok = ok && cudaHostAlloc((void**) &d->input_signal, (size_t) (in_len > 0 ? in_len : 1) * 2, cudaHostAllocDefault) == cudaSuccess;
            ok = ok && cudaHostAlloc((void**) &d->resampled_signal, (size_t) (out_len > 0 ? out_len : 1) * 8, cudaHostAllocDefault) == cudaSuccess;
            ok = ok && cudaMalloc((void**) &d->d_in, (size_t) (in_len > 0 ? in_len : 1) * 2) == cudaSuccess;
            ok = ok && cudaMalloc((void**) &d->d_out, (size_t) (out_len > 0 ? out_len : 1) * 8) == cudaSuccess;
            ok = ok && cudaMalloc((void**) &d->d_tot, 8) == cudaSuccess;
            if (!ok) {
                COMPAT_LOG("rf_decimator_set_parameters: %s", cudaGetErrorString(cudaGetLastError()));
                rf_release_buffers(d);
                d->sample_rate = 0;
                d->down_factor = 0;
                d->input_signal_len = d->resampled_signal_len = 0;
                r = -1;
            } else {
                d->sample_rate = sample_rate;
                d->down_factor = down_factor;
                d->resampled_signal_len = out_len;
                d->input_signal_len = in_len;
            }
            d->surplus = 0;
        }
    }
    pthread_mutex_unlock(&d->mutex);
    return r;
}

// one 100 ms block on the GPU: H2D, boxcar kernel, D2H, integrator write-back (resample.c:6-45)
static int rf_run_block(struct rf_decimator* d)
{
    const size_t in_bytes = (size_t) d->input_signal_len * 2;
    const size_t out_bytes = (size_t) d->resampled_signal_len * 8;
    unsigned int h_tot[2] = {0, 0};
    const unsigned int integ_re = (unsigned int) d->delay.integrator_prev_out.p.re;
    const unsigned int integ_im = (unsigned int) d->delay.integrator_prev_out.p.im;
    const unsigned int comb_re = (unsigned int) d->delay.comb_prev_in.p.re;
    const unsigned int comb_im = (unsigned int) d->delay.comb_prev_in.p.im;
    bool ok = cudaMemcpyAsync(d->d_in, d->input_signal, in_bytes, cudaMemcpyHostToDevice, d->stream) == cudaSuccess;
    ok = ok && cudaMemsetAsync(d->d_tot, 0, 8, d->stream) == cudaSuccess;
    if (ok) {
        int blocks = (d->resampled_signal_len + 255) / 256;
        if (blocks > 1184) blocks = 1184;
        cic_kernel<<<blocks, 256, 0, d->stream>>>((const uint16_t*) d->d_in, d->d_out, d->resampled_signal_len,
                                                  d->down_factor, (int) (integ_re - comb_re), (int) (integ_im - comb_im),
                                                  d->d_tot);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        ok = cudaGetLastError() == cudaSuccess;
    }
    ok = ok && cudaMemcpyAsync(d->resampled_signal, d->d_out, out_bytes, cudaMemcpyDeviceToHost, d->stream) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(h_tot, d->d_tot, 8, cudaMemcpyDeviceToHost, d->stream) == cudaSuccess;
    ok = ok && cudaStreamSynchronize(d->stream) == cudaSuccess;
    if (!ok) return -1;
    d->delay.integrator_prev_out.p.re = (int32_t) (integ_re + h_tot[0]);
    d->delay.integrator_prev_out.p.im = (int32_t) (integ_im + h_tot[1]);
    d->delay.comb_prev_in = d->delay.integrator_prev_out;
    return 0;
}

int rf_decimator_decimate_cmplx_u8(struct rf_decimator* d, const cmplx_u8* complex_signal, int len)
{
    int current_idx = 0;
    int remaining = len;
    int block_size = 0;

    pthread_mutex_lock(&d->mutex);
    block_size = d->input_signal_len - d->surplus;              // rf_decimator.c:88
    if (d->resampled_signal == nullptr || d->input_signal == nullptr || d->input_signal_len <= 0) {   // :90-91
        pthread_mutex_unlock(&d->mutex);      // (the reference returns with the mutex held)
        return -1;
    }
    while (remaining >= block_size) {                            // :93
        memcpy(&d->input_signal[d->surplus], &complex_signal[current_idx], (size_t) block_size * sizeof(cmplx_u8));
        remaining -= block_size;
        current_idx += block_size;
        if (rf_run_block(d)) {                                   // :99-103
            COMPAT_LOG("Error while decimating signal: %s", cudaGetErrorString(cudaGetLastError()));
            pthread_mutex_unlock(&d->mutex);
            return -2;
        }
        for (rf_decimator_callback f : d->callbacks)             // :105, registration order
            f(d->resampled_signal, d->resampled_signal_len);
        d->surplus = 0;                                          // :107-108
        block_size = d->input_signal_len;
    }
    if (remaining > 0) {                                         // :111-115
        memcpy(&d->input_signal[d->surplus], &complex_signal[len - remaining], (size_t) remaining * sizeof(cmplx_u8));
        d->surplus += remaining;
    }
    pthread_mutex_unlock(&d->mutex);
    return 0;
}

void rf_decimator_remove_callbacks(struct rf_decimator* d)
{
    pthread_mutex_lock(&d->mutex);
    d->callbacks.clear();
    pthread_mutex_unlock(&d->mutex);
}

void rf_decimator_free(struct rf_decimator* d)
{
    if (d == nullptr) return;
    rf_decimator_remove_callbacks(d);
    pthread_mutex_destroy(&d->mutex);
    rf_release_buffers(d);
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
}

}  // extern "C"

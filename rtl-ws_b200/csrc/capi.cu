// capi.cu -- the C ABI declared in include/b200sdr.h: argument checking, plans, launches.
// Host code only; every arithmetic step happens in the kernels of this directory.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "b200_common.cuh"
#include "fm_kernels.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

std::atomic<uint64_t> g_launches{0};

static thread_local char t_error[512] = "";

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_error, sizeof(t_error), fmt, ap);
    va_end(ap);
}

int sm_count()
{
    static thread_local int cached_dev = -1;
    static thread_local int cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

namespace {
std::mutex g_attr_mutex;
std::map<std::pair<const void*, int>, int> g_smem_set;          // (kernel, device) -> bytes granted
std::map<std::tuple<const void*, int, int, int>, int> g_occ;     // (kernel, device, block, smem) -> CTAs / SM
}  // namespace

int ensure_dynamic_smem(const void* kernel, int bytes)
{
    int dev = 0;
    B200_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_attr_mutex);
    auto key = std::make_pair(kernel, dev);
    auto it = g_smem_set.find(key);
    if (it != g_smem_set.end() && it->second >= bytes) return B200_OK;
    B200_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    g_smem_set[key] = bytes;
    return B200_OK;
}

int cached_occupancy(const void* kernel, int block_threads, int smem_bytes)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    std::lock_guard<std::mutex> lock(g_attr_mutex);
    auto key = std::make_tuple(kernel, dev, block_threads, smem_bytes);
    auto it = g_occ.find(key);
    if (it != g_occ.end()) return it->second;
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, block_threads, smem_bytes) != cudaSuccess || n < 1) n = 1;
    g_occ[key] = n;
    return n;
}

}  // namespace b200

using namespace b200;

struct b200_spectrum_plan {
    int N;
    int hop;
    int K;
    int64_t row_hop;
    int window;
    int gain_db;
    float db_offset;
    float2* d_twiddle;             // N-point table
    float2* d_twiddle1024;         // 1024-point table (N = 8192 and the four-step sizes run branches of 1024)
    float2* d_twiddle_rk;          // N = 8192: [8][1024] W_N^(r k), the layout spectrum_mx1024.cu reads with immediate offsets
    float2* d_twiddle_4k;          // N = 4096: [64][64] W_4096^(n2 k1), the inter-pass table of spectrum4096.cu
                                   // N = 2048: [32][64] W_2048^(n2 k1), the inter-pass table of spectrum2048.cu
    float* d_window;
    Spec64kExtra x64;              // N = 65536 only (all null otherwise)
    int device;
    // Scratch that belongs to the plan (x64.scratch / x64.acc, and the generic kernel's global work arrays for
    // N > 8192) is shared by every exec of the plan: execs on different CUDA streams are ordered through
    // `scratch_done`, recorded after each launch that touched the scratch and awaited before the next one.
    std::mutex scratch_mutex;
    cudaEvent_t scratch_done;
    bool scratch_used;
    float2* gen_scratch;           // [gen_ctas][2][N] complex, generic kernel, N > 8192
    float* gen_acc;                // [gen_ctas][N]
    int gen_ctas;
};

const float2* b200::spectrum_plan_twiddle(const b200_spectrum_plan* plan) { return plan->d_twiddle; }
float b200::spectrum_plan_db_offset(const b200_spectrum_plan* plan) { return plan->db_offset; }

// Run `launch` (which enqueues a kernel using the plan's scratch on `stream`) after every earlier user of the scratch.
template <class F>
static int with_plan_scratch(b200_spectrum_plan* plan, cudaStream_t stream, F launch)
{
    std::lock_guard<std::mutex> lock(plan->scratch_mutex);
    if (plan->scratch_done == nullptr) B200_CUDA_TRY(cudaEventCreateWithFlags(&plan->scratch_done, cudaEventDisableTiming));
    if (plan->scratch_used) B200_CUDA_TRY(cudaStreamWaitEvent(stream, plan->scratch_done, 0));
    const int rc = launch();
    if (rc != B200_OK) return rc;
    B200_CUDA_TRY(cudaEventRecord(plan->scratch_done, stream));
    plan->scratch_used = true;
    return B200_OK;
}

static float2* upload_twiddles(int N)
{
    std::vector<float2> tw((size_t) N);
    for (int k = 0; k < N; ++k) {
        const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) k / (long double) N;
        tw[k] = make_float2((float) cosl(a), (float) sinl(a));
    }
    float2* d = nullptr;
    if (cudaMalloc(&d, sizeof(float2) * (size_t) N) != cudaSuccess) return nullptr;
    if (cudaMemcpy(d, tw.data(), sizeof(float2) * (size_t) N, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(d);
        return nullptr;
    }
    return d;
}

extern "C" {

int b200_init(int device)
{
    B200_CUDA_TRY(cudaSetDevice(device));
    B200_CUDA_TRY(cudaFree(0));
    cudaDeviceProp prop;
    B200_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("device %d is sm_%d%d; libb200sdr is built for sm_100a only", device, prop.major, prop.minor);
        return B200_ERR_CUDA;
    }
    return B200_OK;
}

const char* b200_last_error(void)
{
    return t_error;
}

uint64_t b200_launch_count(void)
{
    return g_launches.load(std::memory_order_relaxed);
}

int b200_sm_count(void)
{
    return sm_count();
}

// ---- spectrum --------------------------------------------------------------------------

b200_spectrum_plan* b200_spectrum_plan_create(int N, int hop, int K, int64_t row_hop, int window, int gain_db)
{
    if (N < 16 || N > 65536 || (N & (N - 1)) != 0) {
        set_error("spectrum plan: N = %d is not a power of two in [16, 65536]", N);
        return nullptr;
    }
    if (hop <= 0) hop = N;
    if (K < 1) {
        set_error("spectrum plan: K = %d", K);
        return nullptr;
    }
    if (row_hop <= 0) row_hop = (int64_t) K * hop;
    if ((hop % 8) != 0 || (row_hop % 8) != 0) {
        set_error("spectrum plan: hop and row_hop must be multiples of 8 samples");
        return nullptr;
    }
    if (window != B200_WINDOW_RECT && window != B200_WINDOW_HANN) {
        set_error("spectrum plan: unknown window %d", window);
        return nullptr;
    }
    b200_spectrum_plan* pl = new b200_spectrum_plan();
    pl->N = N;
    pl->hop = hop;
    pl->K = K;
    pl->row_hop = row_hop;
    pl->window = window;
    pl->gain_db = gain_db;
    pl->d_twiddle = nullptr;
    pl->d_window = nullptr;
    // cbb_main.c:112: pow(10, gain_db / 10) with the INTEGER quotient; cbb_main.c:125: / count.
    // 2^-14 undoes the (x - 128) / 128 input scale that the kernels leave out of the transform.
    const double g = pow(10.0, (double) (gain_db / 10));
    pl->db_offset = (float) (10.0 * log10(g / ((double) K * 16384.0)));
    if (cudaGetDevice(&pl->device) != cudaSuccess) {
        set_error("spectrum plan: no CUDA device");
        delete pl;
        return nullptr;
    }
    pl->d_twiddle1024 = nullptr;
    pl->d_twiddle_rk = nullptr;
    pl->d_twiddle_4k = nullptr;
    memset(&pl->x64, 0, sizeof(pl->x64));
    pl->scratch_done = nullptr;
    pl->scratch_used = false;
    pl->gen_scratch = nullptr;
    pl->gen_acc = nullptr;
    pl->gen_ctas = 0;
    pl->d_twiddle = upload_twiddles(N);
    const bool four_step = (N == 16384 || N == 32768 || N == 65536);      // spectrum64k.cu, R = N / 1024 branches
    const bool wants1024 = (N == 8192 || four_step);
    if (pl->d_twiddle != nullptr && wants1024) pl->d_twiddle1024 = upload_twiddles(1024);
    if (pl->d_twiddle == nullptr || (wants1024 && pl->d_twiddle1024 == nullptr)) {
        set_error("spectrum plan: twiddle upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (pl->d_twiddle) cudaFree(pl->d_twiddle);
        delete pl;
        return nullptr;
    }
    if (window == B200_WINDOW_HANN) {
        std::vector<float> w((size_t) N);
        for (int i = 0; i < N; ++i)
            w[i] = (float) (0.5L - 0.5L * cosl(2.0L * 3.14159265358979323846264338327950288L * (long double) i /
                                               (long double) N));
        if (cudaMalloc(&pl->d_window, sizeof(float) * (size_t) N) != cudaSuccess ||
            cudaMemcpy(pl->d_window, w.data(), sizeof(float) * (size_t) N, cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("spectrum plan: window upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            cudaFree(pl->d_twiddle);
            if (pl->d_window) cudaFree(pl->d_window);
            delete pl;
            return nullptr;
        }
    }
    if (N == 8192) {
        std::vector<float2> trk((size_t) 8 * 1024);
        for (int r = 0; r < 8; ++r)
            for (int k = 0; k < 1024; ++k) {
                const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) (r * k) / (long double) N;
                trk[(size_t) r * 1024 + k] = make_float2((float) cosl(a), (float) sinl(a));
            }
        if (cudaMalloc((void**) &pl->d_twiddle_rk, sizeof(float2) * trk.size()) != cudaSuccess ||
            cudaMemcpy(pl->d_twiddle_rk, trk.data(), sizeof(float2) * trk.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("spectrum plan: twiddle upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            b200_spectrum_plan_destroy(pl);
            return nullptr;
        }
    }
    if (N == 4096 || N == 2048) {
        const int rows = N / 64;                                    // n2 = 0..rows-1, k1 = 0..63
        std::vector<float2> t4((size_t) rows * 64);
        for (int n2 = 0; n2 < rows; ++n2)
            for (int k1 = 0; k1 < 64; ++k1) {
                const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) (n2 * k1) / (long double) N;
                t4[(size_t) n2 * 64 + k1] = make_float2((float) cosl(a), (float) sinl(a));
            }
        if (cudaMalloc((void**) &pl->d_twiddle_4k, sizeof(float2) * t4.size()) != cudaSuccess ||
            cudaMemcpy(pl->d_twiddle_4k, t4.data(), sizeof(float2) * t4.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("spectrum plan: twiddle upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            b200_spectrum_plan_destroy(pl);
            return nullptr;
        }
    }
    if (four_step) {
        // tables in the layout the four-step kernel reads coalesced, and its L2-resident scratch
        const int Rb = N / 1024;
        std::vector<float2> trk((size_t) Rb * 1024);
        for (int r = 0; r < Rb; ++r)
            for (int k = 0; k < 1024; ++k) {
                const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) ((long long) r * k) / (long double) N;
                trk[(size_t) r * 1024 + k] = make_float2((float) cosl(a), (float) sinl(a));
            }
        bool ok = cudaMalloc((void**) &pl->x64.twiddle_rk, sizeof(float2) * trk.size()) == cudaSuccess &&
                  cudaMemcpy((void*) pl->x64.twiddle_rk, trk.data(), sizeof(float2) * trk.size(), cudaMemcpyHostToDevice) == cudaSuccess;
        pl->x64.scratch_ctas = sm_count();
        ok = ok && cudaMalloc((void**) &pl->x64.scratch, sizeof(float2) * (size_t) N * (size_t) pl->x64.scratch_ctas) == cudaSuccess;
        if (ok && K > 1) ok = cudaMalloc((void**) &pl->x64.acc, sizeof(float) * (size_t) N * (size_t) pl->x64.scratch_ctas) == cudaSuccess;
        if (!ok) {
            set_error("spectrum plan: four-step tables / scratch: %s", cudaGetErrorString(cudaGetLastError()));
            b200_spectrum_plan_destroy(pl);
            return nullptr;
        }
    }
    return pl;
}

void b200_spectrum_plan_destroy(b200_spectrum_plan* plan)
{
    if (plan == nullptr) return;
    if (plan->d_twiddle) cudaFree(plan->d_twiddle);
    if (plan->d_twiddle1024) cudaFree(plan->d_twiddle1024);
    if (plan->d_twiddle_rk) cudaFree(plan->d_twiddle_rk);
    if (plan->d_twiddle_4k) cudaFree(plan->d_twiddle_4k);
    if (plan->d_window) cudaFree(plan->d_window);
    if (plan->x64.twiddle_rk) cudaFree((void*) plan->x64.twiddle_rk);
    if (plan->x64.scratch) cudaFree(plan->x64.scratch);
    if (plan->x64.acc) cudaFree(plan->x64.acc);
    if (plan->gen_scratch) cudaFree(plan->gen_scratch);
    if (plan->gen_acc) cudaFree(plan->gen_acc);
    if (plan->scratch_done) cudaEventDestroy(plan->scratch_done);
    delete plan;
}

int64_t b200_spectrum_plan_rows(const b200_spectrum_plan* plan, int64_t n_samples)
{
    const int64_t span = (int64_t) (plan->K - 1) * plan->hop + plan->N;
    if (n_samples < span) return 0;
    return (n_samples - span) / plan->row_hop + 1;
}

static int spectrum_exec_kind(b200_spectrum_plan* plan, const void* d_in, int64_t stream_stride_bytes, int n_streams,
                              int64_t n_rows, float* d_db, float* d_power, uint8_t* d_db_u8, int kind,
                              void* cuda_stream)
{
    if (plan == nullptr || n_streams < 0 || n_rows < 0) {
        set_error("spectrum exec: bad arguments");
        return B200_ERR_ARG;
    }
    if (n_streams == 0 || n_rows == 0) return B200_OK;
    if (d_in == nullptr) {
        set_error("spectrum exec: null input");
        return B200_ERR_ARG;
    }
    SpecParams p;
    p.iq = reinterpret_cast<const uint8_t*>(d_in);
    p.stream_stride_bytes = stream_stride_bytes;
    p.n_streams = n_streams;
    p.n_rows = n_rows;
    p.hop = plan->hop;
    p.K = plan->K;
    p.row_hop = plan->row_hop;
    p.db = d_db;
    p.power = d_power;
    p.db_u8 = d_db_u8;
    p.db_offset = plan->db_offset;
    p.twiddle = plan->d_twiddle;
    p.twiddle_n = nullptr;
    p.window = plan->d_window;
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (kind == 0 && plan->N == 1024) {
        if ((reinterpret_cast<uintptr_t>(d_in) & 15) != 0 || (stream_stride_bytes & 15) != 0) {
            set_error("spectrum exec: IQ pointer and stream stride must be 16-byte aligned");
            return B200_ERR_ALIGN;
        }
        return launch_spectrum1024(p, stream);
    }
    if (kind == 0 && plan->N >= 2048) {
        if ((reinterpret_cast<uintptr_t>(d_in) & 15) != 0 || (stream_stride_bytes & 15) != 0) {
            set_error("spectrum exec: IQ pointer and stream stride must be 16-byte aligned");
            return B200_ERR_ALIGN;
        }
        if (plan->N == 2048) {
            p.twiddle_n = plan->d_twiddle_4k;
            return launch_spectrum2048(p, stream);
        }
        if (plan->N == 4096) {
            p.twiddle_n = plan->d_twiddle_4k;
            return launch_spectrum4096(p, stream);
        }
        p.twiddle = plan->d_twiddle1024;
        if (plan->N == 8192) {
            p.twiddle_n = plan->d_twiddle_rk;
            return launch_spectrum_mx1024(p, stream);
        }
        return with_plan_scratch(plan, stream, [&] { return launch_spectrum64k(p, plan->x64, plan->N, stream); });
    }
    if (plan->N <= 8192) return launch_spectrum_generic(p, plan->N, kind, nullptr, nullptr, 0, stream);
    // N > 8192 from s32 / f32 input on the generic kernel: its per-CTA work
    // arrays live in the plan, on the plan's device, allocated on first use
    {
        std::lock_guard<std::mutex> lock(plan->scratch_mutex);
        if (plan->gen_scratch == nullptr) {
            int dev = -1;
            B200_CUDA_TRY(cudaGetDevice(&dev));
            if (dev != plan->device) {
                set_error("spectrum exec: the plan was created on device %d, the current device is %d", plan->device, dev);
                return B200_ERR_ARG;
            }
            const int ctas = spectrum_generic_scratch_ctas();
            B200_CUDA_TRY(cudaMalloc(&plan->gen_scratch, (size_t) ctas * 2 * plan->N * sizeof(float2)));
            if (cudaMalloc(&plan->gen_acc, (size_t) ctas * plan->N * sizeof(float)) != cudaSuccess) {
                set_error("spectrum exec: scratch allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
                cudaFree(plan->gen_scratch);
                plan->gen_scratch = nullptr;
                return B200_ERR_CUDA;
            }
            plan->gen_ctas = ctas;
        }
    }
    return with_plan_scratch(plan, stream, [&] {
        return launch_spectrum_generic(p, plan->N, kind, plan->gen_scratch, plan->gen_acc, plan->gen_ctas, stream);
    });
}

int b200_spectrum_exec(b200_spectrum_plan* plan, const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams,
                       int64_t n_rows, float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream)
{
    return spectrum_exec_kind(plan, d_iq, stream_stride_bytes, n_streams, n_rows, d_db, d_power, d_db_u8, 0,
                              cuda_stream);
}

int b200_spectrum_exec_cs32(b200_spectrum_plan* plan, const int32_t* d_iq, int64_t stream_stride_bytes, int n_streams,
                            int64_t n_rows, float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream)
{
    return spectrum_exec_kind(plan, d_iq, stream_stride_bytes, n_streams, n_rows, d_db, d_power, d_db_u8, 1,
                              cuda_stream);
}

int b200_spectrum_exec_rf32(b200_spectrum_plan* plan, const float* d_x, int64_t stream_stride_bytes, int n_streams,
                            int64_t n_rows, float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream)
{
    return spectrum_exec_kind(plan, d_x, stream_stride_bytes, n_streams, n_rows, d_db, d_power, d_db_u8, 2,
                              cuda_stream);
}

// ---- FM branch ---------------------------------------------------------------------------

int b200_fm_history_samples(int R)
{
    return fm_history_samples(R);
}

int b200_fm_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int R, void* cuda_stream)
{
    if (d_iq == nullptr || R < 1 || R > 256 || n_streams < 0) {
        set_error("fm history reset: bad arguments");
        return B200_ERR_ARG;
    }
    return launch_fm_history_reset(d_iq, stream_stride_bytes, n_streams, R, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                          void* cuda_stream)
{
    if (d_iq == nullptr || R < 1 || R > 256 || n_streams < 0) {
        set_error("fm history carry: bad arguments");
        return B200_ERR_ARG;
    }
    return launch_fm_history_carry(d_iq, stream_stride_bytes, n_streams, n_samples, R,
                                   reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_iq_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int history_samples,
                          void* cuda_stream)
{
    if (d_iq == nullptr || n_streams < 0 || history_samples < 8 || history_samples % 8 != 0 ||
        history_samples > B200_IQ_MAX_HISTORY_SAMPLES) {
        set_error("iq history reset: bad arguments (history_samples %d must be a positive multiple of 8, at most 2^30 - 8)", history_samples);
        return B200_ERR_ARG;
    }
    return launch_iq_history_reset(d_iq, stream_stride_bytes, n_streams, history_samples,
                                   reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_iq_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                          int history_samples, void* cuda_stream)
{
    if (d_iq == nullptr || n_streams < 0 || history_samples < 8 || history_samples % 8 != 0 ||
        history_samples > B200_IQ_MAX_HISTORY_SAMPLES) {
        set_error("iq history carry: bad arguments (history_samples %d must be a positive multiple of 8, at most 2^30 - 8)", history_samples);
        return B200_ERR_ARG;
    }
    return launch_iq_history_carry(d_iq, stream_stride_bytes, n_streams, n_samples, history_samples,
                                   reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                 float* d_audio, int64_t audio_stride, int32_t* d_decimated, int64_t dec_stride, void* cuda_stream)
{
    if (d_iq == nullptr || d_audio == nullptr || n_streams < 0) {
        set_error("fm exec: bad arguments");
        return B200_ERR_ARG;
    }
    FmParams p;
    p.iq = d_iq;
    p.stream_stride_bytes = stream_stride_bytes;
    p.n_streams = n_streams;
    p.n_samples = n_samples;
    p.R = R;
    p.audio = d_audio;
    p.audio_stride = audio_stride;
    p.decimated = d_decimated;
    p.dec_stride = dec_stride;
    return launch_fm_chain(p, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_channel_tune(double offset_hz, double sample_rate_hz, uint32_t* phase_inc)
{
    // !(a <= b) also refuses NaN
    if (phase_inc == nullptr || !(sample_rate_hz > 0.0) || !isfinite(sample_rate_hz) ||
        !(fabs(offset_hz) <= 0.5 * sample_rate_hz)) {
        set_error("fm channel tune: offset %g Hz outside +-fs/2 or sample rate %g Hz not positive", offset_hz,
                  sample_rate_hz);
        return B200_ERR_ARG;
    }
    // |offset / fs| <= 1/2, so the rounded value lies in [-2^31, 2^31] and its low 32 bits are the increment
    const int64_t v = (int64_t) llround(offset_hz / sample_rate_hz * 4294967296.0);
    *phase_inc = (uint32_t) (uint64_t) v;
    return B200_OK;
}

int b200_fm_channels_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                          int64_t first_sample, const uint32_t* d_phase_inc, int n_channels, float* d_audio,
                          int64_t audio_stride, float* d_baseband, int64_t baseband_stride, void* cuda_stream)
{
    return launch_fm_channels(d_iq, stream_stride_bytes, n_streams, n_samples, R, first_sample, d_phase_inc,
                              n_channels, d_audio, audio_stride, d_baseband, baseband_stride, nullptr, 0,
                              reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_channel_filter_design(int R, int n_taps, double cutoff_hz, double atten_db, double sample_rate_hz,
                                  float* h_taps)
{
    return fm_channel_filter_design(R, n_taps, cutoff_hz, atten_db, sample_rate_hz, h_taps);
}

int b200_fm_channels_fir_history_samples(int R, int n_taps)
{
    const int h = fm_channels_fir_history_samples(R, n_taps);
    if (h < 0) set_error("fm channels fir history: R %d or %d taps out of range", R, n_taps);
    return h;
}

int b200_fm_channels_exec_fir(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                              int64_t first_sample, const uint32_t* d_phase_inc, int n_channels, float* d_audio,
                              int64_t audio_stride, float* d_baseband, int64_t baseband_stride, const float* d_taps,
                              int n_taps, void* cuda_stream)
{
    if (d_taps == nullptr && n_taps == 0) {        // launch_fm_channels would take it for the boxcar
        set_error("fm channels fir: no taps");
        return B200_ERR_ARG;
    }
    return launch_fm_channels(d_iq, stream_stride_bytes, n_streams, n_samples, R, first_sample, d_phase_inc,
                              n_channels, d_audio, audio_stride, d_baseband, baseband_stride, d_taps, n_taps,
                              reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_channels_exec_runs(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                               int R, const b200_fm_channel_run* h_runs, int n_runs, float* d_audio,
                               int64_t audio_stride, int64_t n_audio_rows, const float* d_taps, int n_taps,
                               void* cuda_stream)
{
    return launch_fm_channels_runs(d_iq, stream_stride_bytes, n_streams, n_samples, R, h_runs, n_runs, d_audio,
                                   audio_stride, n_audio_rows, d_taps, n_taps, reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- pinned host memory --------------------------------------------------------------------

void* b200_host_alloc(uint64_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, (size_t) bytes, cudaHostAllocDefault) != cudaSuccess) {
        set_error("b200_host_alloc(%llu): %s", (unsigned long long) bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}

void b200_host_free(void* p)
{
    if (p != nullptr) cudaFreeHost(p);
}

}  // extern "C"

// capi.cu -- the C ABI declared in include/b200sdr.h: argument checking, plans, launches.
// Host code only; every arithmetic step happens in the kernels of this directory.
#include <math.h>
#include <stdarg.h>

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
    int N = 0;
    int hop = 0;
    int K = 0;
    int64_t row_hop = 0;
    float db_offset = 0.0f;
    int device = -1;
    float2* d_twiddle = nullptr;        // N-point table
    float2* d_twiddle1024 = nullptr;    // 1024-point table: from N = 8192 up the u8 kernels run transforms of 1024 points
    float2* d_twiddle_pass = nullptr;   // from N = 2048 up, the inter-pass table [N / C][C] = W_N^(r c) of the u8 kernels:
                                        // C = 64 below N = 8192, else 1024
    float* d_window = nullptr;
    int four_step_ctas = 0;             // N > 8192: the grid of the four-step kernel (u8) and of the generic kernel's
    int generic_ctas = 0;               // global-scratch form (cs32 / rf32)
    // Scratch shared by every exec of the plan, grow-only: [four_step_ctas][N] complex + [four_step_ctas][N] floats
    // (K > 1) for the four-step kernel, reserved at creation; [generic_ctas][2][N] complex + [generic_ctas][N] floats
    // for the generic kernel, grown on its first exec.  Execs on different CUDA streams are ordered through
    // `scratch_done`, recorded after each launch that used the scratch and awaited before the next one.
    std::mutex scratch_mutex;
    cudaEvent_t scratch_done = nullptr;
    bool scratch_used = false;
    float2* work = nullptr;
    size_t work_n = 0;
    float* acc = nullptr;
    size_t acc_n = 0;
};

const float2* b200::spectrum_plan_twiddle(const b200_spectrum_plan* plan) { return plan->d_twiddle; }
float b200::spectrum_plan_db_offset(const b200_spectrum_plan* plan) { return plan->db_offset; }

// Grow the plan's scratch to at least `work` complex and `acc` float entries.  The caller holds scratch_mutex or is
// the plan's only user.
static cudaError_t grow_scratch(b200_spectrum_plan* plan, size_t work, size_t acc)
{
    if (work <= plan->work_n && acc <= plan->acc_n) return cudaSuccess;
    // an exec on another CUDA stream may still be reading the buffers this frees
    if (plan->scratch_used)
        if (cudaError_t e = cudaEventSynchronize(plan->scratch_done)) return e;
    auto grow = [](auto*& buf, size_t& have, size_t want) {
        if (want <= have) return cudaSuccess;
        cudaFree(buf);
        buf = nullptr;
        have = 0;
        if (cudaError_t e = cudaMalloc(&buf, want * sizeof(*buf))) {
            buf = nullptr;
            return e;
        }
        have = want;
        return cudaSuccess;
    };
    if (cudaError_t e = grow(plan->work, plan->work_n, work)) return e;
    return grow(plan->acc, plan->acc_n, acc);
}

// Run `launch` (which enqueues a kernel using the plan's scratch on `stream`) with the scratch grown to at least `work`
// complex and `acc` float entries, after every earlier user of the scratch.
template <class F>
static int launch_with_scratch(b200_spectrum_plan* plan, size_t work, size_t acc, cudaStream_t stream, F launch)
{
    std::lock_guard<std::mutex> lock(plan->scratch_mutex);
    if (work > plan->work_n || acc > plan->acc_n) {
        int dev = -1;
        B200_CUDA_TRY(cudaGetDevice(&dev));
        if (dev != plan->device) {
            set_error("spectrum exec: the plan was created on device %d, the current device is %d", plan->device, dev);
            return B200_ERR_ARG;
        }
        if (cudaError_t e = grow_scratch(plan, work, acc)) {
            set_error("spectrum exec: scratch allocation failed: %s", cudaGetErrorString(e));
            return B200_ERR_CUDA;
        }
    }
    if (plan->scratch_done == nullptr) B200_CUDA_TRY(cudaEventCreateWithFlags(&plan->scratch_done, cudaEventDisableTiming));
    if (plan->scratch_used) B200_CUDA_TRY(cudaStreamWaitEvent(stream, plan->scratch_done, 0));
    const int rc = launch();
    if (rc != B200_OK) return rc;
    B200_CUDA_TRY(cudaEventRecord(plan->scratch_done, stream));
    plan->scratch_used = true;
    return B200_OK;
}

constexpr long double PI_L = 3.14159265358979323846264338327950288L;

// A new device copy of `h`, or null.
template <class T>
static T* upload(const std::vector<T>& h)
{
    T* d = nullptr;
    if (cudaMalloc(&d, sizeof(T) * h.size()) != cudaSuccess) return nullptr;
    if (cudaMemcpy(d, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(d);
        return nullptr;
    }
    return d;
}

// The N entries W_N^e(i) = exp(-2 pi i e(i) / N), i = 0..N-1, computed in long double and rounded to float.
template <class E>
static float2* upload_twiddles(int N, E e)
{
    std::vector<float2> tw((size_t) N);
    for (int i = 0; i < N; ++i) {
        const long double a = -2.0L * PI_L * (long double) e(i) / (long double) N;
        tw[i] = make_float2((float) cosl(a), (float) sinl(a));
    }
    return upload(tw);
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
    int device = -1;
    if (cudaGetDevice(&device) != cudaSuccess) {
        set_error("spectrum plan: no CUDA device");
        return nullptr;
    }
    b200_spectrum_plan* pl = new b200_spectrum_plan();
    pl->N = N;
    pl->hop = hop;
    pl->K = K;
    pl->row_hop = row_hop;
    pl->device = device;
    // cbb_main.c:112: pow(10, gain_db / 10) with the INTEGER quotient; cbb_main.c:125: / count.
    // 2^-14 undoes the (x - 128) / 128 input scale that the kernels leave out of the transform.
    const double g = pow(10.0, (double) (gain_db / 10));
    pl->db_offset = (float) (10.0 * log10(g / ((double) K * 16384.0)));
    auto fail = [pl](const char* what) -> b200_spectrum_plan* {
        set_error("spectrum plan: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
        b200_spectrum_plan_destroy(pl);
        return nullptr;
    };
    const auto identity = [](int64_t i) { return i; };
    if ((pl->d_twiddle = upload_twiddles(N, identity)) == nullptr) return fail("twiddle upload failed");
    if (N >= 8192 && (pl->d_twiddle1024 = upload_twiddles(1024, identity)) == nullptr) return fail("twiddle upload failed");
    if (N >= 2048) {
        const int64_t C = N >= 8192 ? 1024 : 64;
        pl->d_twiddle_pass = upload_twiddles(N, [C](int64_t i) { return (i / C) * (i % C); });
        if (pl->d_twiddle_pass == nullptr) return fail("twiddle upload failed");
    }
    if (window == B200_WINDOW_HANN) {
        std::vector<float> w((size_t) N);
        for (int i = 0; i < N; ++i) w[i] = (float) (0.5L - 0.5L * cosl(2.0L * PI_L * (long double) i / (long double) N));
        if ((pl->d_window = upload(w)) == nullptr) return fail("window upload failed");
    }
    if (N > 8192) {
        pl->four_step_ctas = sm_count();
        pl->generic_ctas = spectrum_generic_scratch_ctas();
        const size_t slice = (size_t) pl->four_step_ctas * N;
        if (grow_scratch(pl, slice, K > 1 ? slice : 0) != cudaSuccess) return fail("scratch allocation failed");
    }
    return pl;
}

void b200_spectrum_plan_destroy(b200_spectrum_plan* plan)
{
    if (plan == nullptr) return;
    for (void* d : std::initializer_list<void*>{plan->d_twiddle, plan->d_twiddle1024, plan->d_twiddle_pass, plan->d_window,
                                                plan->work, plan->acc})
        if (d != nullptr) cudaFree(d);
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
    const int N = plan->N;
    // u8 input from 1024 points up runs a kernel made for its N, which reads 16-byte words; the rest runs the generic one
    const bool specialised = kind == 0 && N >= 1024;
    if (specialised && ((reinterpret_cast<uintptr_t>(d_in) & 15) != 0 || (stream_stride_bytes & 15) != 0)) {
        set_error("spectrum exec: IQ pointer and stream stride must be 16-byte aligned");
        return B200_ERR_ALIGN;
    }
    const uint64_t total = (uint64_t) n_streams * (uint64_t) n_rows;
    if (specialised && N <= 8192 && total >= (1ull << 31)) {         // these four index rows in 32 bits
        set_error("spectrum: n_streams * n_rows = %llu exceeds 2^31 - 1 rows per launch", (unsigned long long) total);
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
    p.twiddle = specialised && N >= 8192 ? plan->d_twiddle1024 : plan->d_twiddle;
    p.twiddle_n = specialised ? plan->d_twiddle_pass : nullptr;
    p.window = plan->d_window;
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (!specialised) {
        if (N <= 8192) return launch_spectrum_generic(p, N, kind, nullptr, nullptr, 0, stream);
        const size_t ctas = (size_t) plan->generic_ctas;
        return launch_with_scratch(plan, ctas * 2 * N, ctas * N, stream, [&] {
            return launch_spectrum_generic(p, N, kind, plan->work, plan->acc, plan->generic_ctas, stream);
        });
    }
    switch (N) {
    case 1024: return launch_spectrum1024(p, stream);
    case 2048: return launch_spectrum2048(p, stream);
    case 4096: return launch_spectrum4096(p, stream);
    case 8192: return launch_spectrum_mx1024(p, stream);
    }
    const size_t slice = (size_t) plan->four_step_ctas * N;
    return launch_with_scratch(plan, slice, plan->K > 1 ? slice : 0, stream, [&] {
        const Spec64kExtra x = {plan->work, plan->K > 1 ? plan->acc : nullptr, plan->d_twiddle_pass, plan->four_step_ctas};
        return launch_spectrum64k(p, x, N, stream);
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

// The checks the four history calls share.  The FM calls pass 32 R, or 0 for a down factor outside [1, 256].
static bool history_args_ok(const char* who, const uint8_t* d_iq, int n_streams, int history_samples)
{
    if (d_iq != nullptr && n_streams >= 0 && history_samples >= 8 && history_samples % 8 == 0 &&
        history_samples <= B200_IQ_MAX_HISTORY_SAMPLES)
        return true;
    set_error("%s: bad arguments (IQ %p, %d streams, a history of %d samples: it must be a positive multiple of 8, "
              "at most 2^30 - 8)", who, (const void*) d_iq, n_streams, history_samples);
    return false;
}

int b200_fm_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int R, void* cuda_stream)
{
    const int h = R >= 1 && R <= 256 ? fm_history_samples(R) : 0;
    if (!history_args_ok("fm history reset", d_iq, n_streams, h)) return B200_ERR_ARG;
    return launch_iq_history_reset(d_iq, stream_stride_bytes, n_streams, h, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_fm_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                          void* cuda_stream)
{
    const int h = R >= 1 && R <= 256 ? fm_history_samples(R) : 0;
    if (!history_args_ok("fm history carry", d_iq, n_streams, h)) return B200_ERR_ARG;
    return launch_iq_history_carry(d_iq, stream_stride_bytes, n_streams, n_samples, h,
                                   reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_iq_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int history_samples,
                          void* cuda_stream)
{
    if (!history_args_ok("iq history reset", d_iq, n_streams, history_samples)) return B200_ERR_ARG;
    return launch_iq_history_reset(d_iq, stream_stride_bytes, n_streams, history_samples,
                                   reinterpret_cast<cudaStream_t>(cuda_stream));
}

int b200_iq_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                          int history_samples, void* cuda_stream)
{
    if (!history_args_ok("iq history carry", d_iq, n_streams, history_samples)) return B200_ERR_ARG;
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

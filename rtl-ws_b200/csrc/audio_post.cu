// audio_post.cu -- opt-in audio extensions behind the FM branch (sm_100a): single-pole de-emphasis
// and a 15/16 polyphase resampler, 51.2 kHz -> 48 kHz.
//
// NEITHER exists in the reference: its chain ends at fs / (4R) = 51.2 kS/s float audio with no
// de-emphasis (audio_main.c:133-139, rf_decimator.c:65-66), while its own UI insists on a 48 kHz
// AudioContext (resources/rtl_ui.js:79-82) and plays the 51.2 kHz stream 6 % slow.  BASELINE.json's north
// star names "de-emphasis and resampler ... 48 kHz audio", so both are offered as extensions that are
// OFF by default: without flags nothing in this file runs and every output bit is the reference's.
// The definitions (the test oracle restates them as plain sequential loops):
//
//   de-emphasis   y[n] = y[n-1] + alpha * (x[n] - y[n-1]),  alpha = 1 - exp(-1 / (rate * tau)),
//                 tau = 50 us (B200_AUDIO_DEEMPH_50US, Europe) or 75 us (.._75US, Americas), y[-1] = 0
//   resampler     y[m] = sum_{t=0}^{15} h[r + 15 t] * x[q - t],  q = floor(16 m / 15), r = 16 m mod 15,
//                 h = 240-tap Blackman-windowed sinc, cutoff 24 kHz at the 768 kHz interpolated rate,
//                 DC gain 15 (unity per phase); x[<0] = 0.  16 input samples -> 15 output samples.
//
// The recursion is a scan, but a short-memory one: a thread that starts L samples early from y = 0 is off
// by at most (1 - alpha)^L times the signal's peak, so the host picks the run-in
//   L = max(96, ceil(ln(1e-7) / ln(1 - alpha)) rounded up to a multiple of 8)
// and the result matches the sequential one within f32 rounding.  At the reference's 51.2 kHz L is 96 for both
// time constants ((1 - alpha)^96 < 2e-11 there); alpha shrinks as the rate grows, so L grows with it: 312 at
// 256 kHz and 624 at 512 kHz with 75 us.  De-emphasis is refused when L would exceed AP_MAX_RUNIN (above about
// 850 kHz at 75 us and 1.27 MHz at 50 us).  Each thread produces 8 samples after its run-in; only a batch's
// first samples use the carried y[-1] itself.  At 51.2 kHz the audio is 1/40 of the input sample rate (0.1 B
// per input sample), so this pass costs nothing next to the chain kernel.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <mutex>

#include "b200_common.cuh"

namespace b200 {

namespace {

constexpr int AP_PER_THREAD = 8;
constexpr int AP_CHUNK = 1024;                 // input samples per CTA
constexpr int AP_HALO = 16;                    // e[] samples in front of the chunk (15 needed)
constexpr int AP_THREADS = 160;                // >= (AP_CHUNK + AP_HALO) / AP_PER_THREAD = 130
constexpr int AP_MIN_RUNIN = 96;
constexpr int AP_MAX_RUNIN = 1024;
constexpr int AP_TAPS = 240;
constexpr int AP_T = 16;                       // taps per phase

// state layout, floats: [0] y[-1] of the de-emphasis, [1..15] the last 15 resampler inputs (oldest first),
// [32..47] staging written by the last chunk, committed by audio_post_commit_kernel
constexpr int APS_Y = 0;
constexpr int APS_HIST = 1;
constexpr int APS_NEXT = 32;
static_assert(B200_AUDIO_POST_STATE_FLOATS >= APS_NEXT + 16, "audio post state");

__constant__ float c_resample_taps[AP_TAPS];

struct PostParams {
    const float* in;
    int64_t in_stride;
    int64_t n;                  // input samples per stream
    float* out;
    int64_t out_stride;
    float* state;               // [n_streams][B200_AUDIO_POST_STATE_FLOATS]
    float alpha;                // 0 = no de-emphasis
    int runin;                  // de-emphasis samples each thread runs before its first output
    int resample;
};

// One chunk (blockIdx.x) of one row (blockIdx.y).  ROWS: the row names its input, output and state rows and
// whether it is fresh, i.e. reads the state as all zero (stream start) without touching it; otherwise all three are
// row blockIdx.y and the state is read.  The next state is staged in the state row's [APS_NEXT..] either way.
template <bool ROWS>
__device__ __forceinline__ void audio_post_chunk(const PostParams& p, const b200_audio_post_row* rows)
{
    __shared__ float e[AP_CHUNK + AP_HALO];      // e[i] = de-emphasised sample c0 - 16 + i
    __shared__ float taps[AP_TAPS];              // lanes read different phases: shared memory, not the constant port
    const int tid = threadIdx.x;
    if (p.resample)
        for (int i = tid; i < AP_TAPS; i += AP_THREADS) taps[i] = c_resample_taps[i];
    const int s = blockIdx.y;
    const int64_t c0 = (int64_t) blockIdx.x * AP_CHUNK;
    const int n_here = (int) min((int64_t) AP_CHUNK, p.n - c0);
    const float* x = p.in + (int64_t) (ROWS ? rows[s].audio_row : s) * p.in_stride;
    float* st = p.state + (int64_t) (ROWS ? rows[s].state_row : s) * B200_AUDIO_POST_STATE_FLOATS;
    const bool fresh = ROWS && rows[s].fresh != 0;
    const bool last = c0 + n_here == p.n;

    // ---- de-emphasis (or a plain copy) of samples [c0 - 16, c0 + n_here) into e[] ----
    {
        const int i0 = tid * AP_PER_THREAD;                         // index into e[]
        const int64_t g0 = c0 - AP_HALO + i0;                       // first global sample of this thread
        if (i0 < n_here + AP_HALO) {
            if (p.alpha > 0.0f) {
                float y;
                int64_t g = g0 - p.runin;
                if (g <= 0) {                                       // the run-in would cross the batch start: exact state
                    y = fresh ? 0.0f : st[APS_Y];
                    g = 0;
                } else {
                    y = 0.0f;
                }
                // samples before the batch (only the first chunk's halo threads see them) come from the state
                for (; g < g0; ++g) y = fmaf(p.alpha, x[g] - y, y);
#pragma unroll
                for (int k = 0; k < AP_PER_THREAD; ++k) {
                    const int64_t gg = g0 + k;
                    if (i0 + k < n_here + AP_HALO) {
                        if (gg >= 0) {
                            y = fmaf(p.alpha, x[gg] - y, y);
                            e[i0 + k] = y;
                        } else {
                            e[i0 + k] = gg >= -15 && !fresh ? st[APS_HIST + 15 + (int) gg] : 0.0f;
                        }
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < AP_PER_THREAD; ++k) {
                    const int64_t gg = g0 + k;
                    if (i0 + k < n_here + AP_HALO)
                        e[i0 + k] = gg >= 0 ? x[gg] : (gg >= -15 && !fresh ? st[APS_HIST + 15 + (int) gg] : 0.0f);
                }
            }
        }
    }
    __syncthreads();

    // ---- output ----
    float* out = p.out + (int64_t) (ROWS ? rows[s].out_row : s) * p.out_stride;
    if (p.resample) {
        const int n_out = n_here / 16 * 15;                         // n is a multiple of 16
        const int64_t m0 = c0 / 16 * 15;
        for (int j = tid; j < n_out; j += AP_THREADS) {
            const int q = (16 * j) / 15;                            // chunk-local input index (c0 is a multiple of 16)
            const int r = 16 * j - 15 * q;
            const float* xe = e + AP_HALO + q;
            float acc = 0.0f;
#pragma unroll
            for (int t = 0; t < AP_T; ++t) acc = fmaf(taps[r + 15 * t], xe[-t], acc);
            out[m0 + j] = acc;
        }
    } else {
        for (int i = tid; i < n_here; i += AP_THREADS) out[c0 + i] = e[AP_HALO + i];
    }

    // ---- next state (staged; the first chunk of this launch may still be reading the current one) ----
    if (last && tid < 16) {
        // e[] holds at least 16 + n_here valid entries; a batch shorter than 15 keeps old history in front
        st[APS_NEXT + tid] = tid == 0 ? e[AP_HALO + n_here - 1] : e[AP_HALO + n_here - 16 + tid];
    }
}

__global__ void __launch_bounds__(AP_THREADS) audio_post_kernel(const PostParams p)
{
    audio_post_chunk<false>(p, nullptr);
}

// The row table of b200_audio_post_rows, passed by value like FcRunsParams: 16 B a row, 16 KB in all
struct PostRowsParams : PostParams {
    b200_audio_post_row rows[B200_AUDIO_POST_MAX_ROWS];
};

__global__ void __launch_bounds__(AP_THREADS) audio_post_rows_kernel(const __grid_constant__ PostRowsParams p)
{
    audio_post_chunk<true>(p, p.rows);
}

__global__ void audio_post_commit_kernel(float* state, int n_streams)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_streams * 16) return;
    float* st = state + (int64_t) (i / 16) * B200_AUDIO_POST_STATE_FLOATS;
    st[i % 16] = st[APS_NEXT + i % 16];
}

// the commit of the table's state rows (no two rows share one)
__global__ void audio_post_commit_rows_kernel(const __grid_constant__ PostRowsParams p, int n_rows)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * 16) return;
    float* st = p.state + (int64_t) p.rows[i / 16].state_row * B200_AUDIO_POST_STATE_FLOATS;
    st[i % 16] = st[APS_NEXT + i % 16];
}

std::mutex g_taps_mutex;
bool g_taps_uploaded[64] = {false};

}  // namespace

// The 240-tap prototype, in double, rounded to float once (the test oracle evaluates the same statements)
void audio_resample_taps(float* h)
{
    const double pi = 3.14159265358979323846;
    const double fc = 1.0 / 32.0;                   // cycles per interpolated sample: 24 kHz of 768 kHz
    const double mid = (AP_TAPS - 1) / 2.0;
    double w[AP_TAPS];
    double sum = 0.0;
    for (int k = 0; k < AP_TAPS; ++k) {
        const double t = (double) k - mid;
        const double a = 2.0 * pi * fc * t;
        const double sinc = t == 0.0 ? 1.0 : sin(a) / a;
        const double win = 0.42 - 0.5 * cos(2.0 * pi * (double) k / (AP_TAPS - 1)) + 0.08 * cos(4.0 * pi * (double) k / (AP_TAPS - 1));
        w[k] = sinc * win;
        sum += w[k];
    }
    for (int k = 0; k < AP_TAPS; ++k) h[k] = (float) (w[k] * 15.0 / sum);
}

static int ensure_taps()
{
    int dev = 0;
    B200_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_taps_mutex);
    if (dev < 64 && g_taps_uploaded[dev]) return B200_OK;
    float h[AP_TAPS];
    audio_resample_taps(h);
    B200_CUDA_TRY(cudaMemcpyToSymbol(c_resample_taps, h, sizeof(h)));
    if (dev < 64) g_taps_uploaded[dev] = true;
    return B200_OK;
}

// The flag, rate and length rules every audio post path shares; alpha and runin (nullable) receive the kernel's
// de-emphasis coefficient (0 = none) and run-in.
int audio_post_check(const char* who, int flags, double audio_rate_hz, int64_t n_audio, float* alpha, int* runin)
{
    const int de = flags & (B200_AUDIO_DEEMPH_50US | B200_AUDIO_DEEMPH_75US);
    if (n_audio < 0 || de == (B200_AUDIO_DEEMPH_50US | B200_AUDIO_DEEMPH_75US) || (flags & ~7) != 0 ||
        !(audio_rate_hz > 0.0)) {
        set_error("%s: bad arguments (flags = %d)", who, flags);
        return B200_ERR_ARG;
    }
    if ((flags & B200_AUDIO_RESAMPLE_48K) && n_audio % 16 != 0) {
        set_error("%s: the 15/16 resampler takes multiples of 16 samples, not %lld", who, (long long) n_audio);
        return B200_ERR_ARG;
    }
    float a = 0.0f;
    int L = AP_MIN_RUNIN;
    if (de) {
        const double tau = de == B200_AUDIO_DEEMPH_50US ? 50e-6 : 75e-6;
        a = (float) (1.0 - exp(-1.0 / (audio_rate_hz * tau)));
        // run-in after which a start from y = 0 is off by (1 - alpha)^L <= 1e-7 of the signal's peak (alpha = 0,
        // a rate so high that alpha rounds away, would need an endless one)
        const double need = ceil(log(1e-7) / log1p(-(double) a));
        if (!(a > 0.0f) || !(need <= AP_MAX_RUNIN)) {
            set_error("%s: de-emphasis at %g Hz needs a run-in of %g samples, more than %d", who, audio_rate_hz, need,
                      AP_MAX_RUNIN);
            return B200_ERR_ARG;
        }
        L = (int) need > AP_MIN_RUNIN ? ((int) need + 7) / 8 * 8 : AP_MIN_RUNIN;
    }
    if (alpha) *alpha = a;
    if (runin) *runin = L;
    return B200_OK;
}

}  // namespace b200

using namespace b200;

// bytes from the first float of `rows` rows `stride` floats apart to one past the last of the last row's `width`
// floats; -1 for no rows or an extent past int64
static int64_t block_bytes(int64_t rows, int64_t stride, int64_t width)
{
    if (rows < 1 || stride < 0 || width < 0 || width > INT64_MAX / 8) return -1;
    if (stride > 0 && rows - 1 > (INT64_MAX / 4 - width) / stride) return -1;
    return ((rows - 1) * stride + width) * 4;
}

static bool overlap(const void* a, int64_t a_bytes, const void* b, int64_t b_bytes)
{
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + (uintptr_t) b_bytes && y < x + (uintptr_t) a_bytes;
}

extern "C" {

int64_t b200_audio_post_out_samples(int64_t n_audio, int flags)
{
    if (n_audio < 0) return B200_ERR_ARG;
    if (flags & B200_AUDIO_RESAMPLE_48K) return n_audio % 16 == 0 ? n_audio / 16 * 15 : B200_ERR_ARG;
    return n_audio;
}

int b200_audio_resample_taps(float* h240)
{
    if (h240 == nullptr) return B200_ERR_ARG;
    audio_resample_taps(h240);
    return AP_TAPS;
}

int b200_audio_post(const float* d_audio, int64_t audio_stride, int n_streams, int64_t n_audio, double audio_rate_hz,
                    int flags, float* d_state, float* d_out, int64_t out_stride, void* cuda_stream)
{
    PostParams p;
    if (d_audio == nullptr || d_out == nullptr || d_state == nullptr || n_streams < 0) {
        set_error("audio post: bad arguments (flags = %d)", flags);
        return B200_ERR_ARG;
    }
    if (int rc = audio_post_check("audio post", flags, audio_rate_hz, n_audio, &p.alpha, &p.runin)) return rc;
    if (n_streams == 0 || n_audio == 0) return B200_OK;
    if (n_streams > 65535 || (n_audio + AP_CHUNK - 1) / AP_CHUNK >= (1ll << 31)) {
        set_error("audio post: too large for one launch");
        return B200_ERR_ARG;
    }
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    p.in = d_audio;
    p.in_stride = audio_stride;
    p.n = n_audio;
    p.out = d_out;
    p.out_stride = out_stride;
    p.state = d_state;
    p.resample = (flags & B200_AUDIO_RESAMPLE_48K) != 0;
    if (p.resample)
        if (int rc = ensure_taps()) return rc;
    const unsigned chunks = (unsigned) ((n_audio + AP_CHUNK - 1) / AP_CHUNK);
    audio_post_kernel<<<dim3(chunks, (unsigned) n_streams), AP_THREADS, 0, stream>>>(p);
    B200_LAUNCH_CHECK();
    audio_post_commit_kernel<<<(n_streams * 16 + 255) / 256, 256, 0, stream>>>(d_state, n_streams);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

int b200_audio_post_rows(const float* d_audio, int64_t audio_stride, int64_t n_audio_rows, int64_t n_audio,
                         double audio_rate_hz, int flags, const b200_audio_post_row* h_rows, int n_rows,
                         float* d_state, int64_t n_state_rows, float* d_out, int64_t out_stride, int64_t n_out_rows,
                         void* cuda_stream)
{
    static thread_local PostRowsParams p;        // 16 KB: kept off the caller's stack
    if (d_audio == nullptr || d_out == nullptr || d_state == nullptr || h_rows == nullptr || n_rows < 1 ||
        n_rows > B200_AUDIO_POST_MAX_ROWS) {
        set_error("audio post rows: null pointer or %d rows outside [1, %d]", n_rows, B200_AUDIO_POST_MAX_ROWS);
        return B200_ERR_ARG;
    }
    if (int rc = audio_post_check("audio post rows", flags, audio_rate_hz, n_audio, &p.alpha, &p.runin)) return rc;
    const int64_t n_out = b200_audio_post_out_samples(n_audio, flags);
    // the byte extent of each block: rows past its stride would overlap and race
    const int64_t in_bytes = block_bytes(n_audio_rows, audio_stride, n_audio);
    const int64_t out_bytes = block_bytes(n_out_rows, out_stride, n_out);
    const int64_t state_bytes = block_bytes(n_state_rows, B200_AUDIO_POST_STATE_FLOATS, B200_AUDIO_POST_STATE_FLOATS);
    if (audio_stride < n_audio || out_stride < n_out || in_bytes < 0 || out_bytes < 0 || state_bytes < 0) {
        set_error("audio post rows: %lld input rows %lld floats apart for %lld samples, %lld output rows %lld apart for "
                  "%lld, %lld state rows", (long long) n_audio_rows, (long long) audio_stride, (long long) n_audio,
                  (long long) n_out_rows, (long long) out_stride, (long long) n_out, (long long) n_state_rows);
        return B200_ERR_ARG;
    }
    if (((reinterpret_cast<uintptr_t>(d_audio) | reinterpret_cast<uintptr_t>(d_out) |
          reinterpret_cast<uintptr_t>(d_state)) & 3) != 0) {
        set_error("audio post rows: audio, state and output must be 4-byte aligned");
        return B200_ERR_ALIGN;
    }
    if (overlap(d_out, out_bytes, d_audio, in_bytes) || overlap(d_state, state_bytes, d_audio, in_bytes) ||
        overlap(d_state, state_bytes, d_out, out_bytes)) {
        set_error("audio post rows: the audio, output and state blocks may not overlap");
        return B200_ERR_ARG;
    }
    int32_t out_rows[B200_AUDIO_POST_MAX_ROWS], state_rows[B200_AUDIO_POST_MAX_ROWS];
    for (int k = 0; k < n_rows; ++k) {
        const b200_audio_post_row& r = h_rows[k];
        if (r.audio_row < 0 || r.audio_row >= n_audio_rows || r.out_row < 0 || r.out_row >= n_out_rows ||
            r.state_row < 0 || r.state_row >= n_state_rows) {
            set_error("audio post rows: row %d (audio row %d of %lld, output row %d of %lld, state row %d of %lld)", k,
                      r.audio_row, (long long) n_audio_rows, r.out_row, (long long) n_out_rows, r.state_row,
                      (long long) n_state_rows);
            return B200_ERR_ARG;
        }
        out_rows[k] = r.out_row;
        state_rows[k] = r.state_row;
    }
    // two rows writing one output row or one state row would race
    std::sort(out_rows, out_rows + n_rows);
    std::sort(state_rows, state_rows + n_rows);
    for (int k = 1; k < n_rows; ++k)
        if (out_rows[k] == out_rows[k - 1] || state_rows[k] == state_rows[k - 1]) {
            set_error("audio post rows: two rows share output row %d or state row %d", out_rows[k], state_rows[k]);
            return B200_ERR_ARG;
        }
    if (n_audio == 0) return B200_OK;
    if ((n_audio + AP_CHUNK - 1) / AP_CHUNK >= (1ll << 31)) {
        set_error("audio post rows: too large for one launch");
        return B200_ERR_ARG;
    }
    p.in = d_audio;
    p.in_stride = audio_stride;
    p.n = n_audio;
    p.out = d_out;
    p.out_stride = out_stride;
    p.state = d_state;
    p.resample = (flags & B200_AUDIO_RESAMPLE_48K) != 0;
    memcpy(p.rows, h_rows, sizeof(b200_audio_post_row) * (size_t) n_rows);
    if (p.resample)
        if (int rc = ensure_taps()) return rc;
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    const unsigned chunks = (unsigned) ((n_audio + AP_CHUNK - 1) / AP_CHUNK);
    audio_post_rows_kernel<<<dim3(chunks, (unsigned) n_rows), AP_THREADS, 0, stream>>>(p);
    B200_LAUNCH_CHECK();
    audio_post_commit_rows_kernel<<<(n_rows * 16 + 255) / 256, 256, 0, stream>>>(p, n_rows);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // extern "C"

// chain.cu -- the full spectrum + FM chain entry points (b200sdr.h): device-resident
// b200_chain_exec and the host-buffer session that wraps it with pipelined PCIe copies.
#include <mutex>
#include <map>

#include "b200_common.cuh"
#include "fm_kernels.cuh"
#include "spectrum_kernels.cuh"

using namespace b200;

namespace {

constexpr int CHAIN_N = 1024;      // cbb_main.c:17 FFT_POINTS
constexpr int CHAIN_R = 10;        // cbb_main.c:80 at rtl_sensor.c:12's 2.048 MS/s and main.c:23's 192 kHz
constexpr int CHAIN_TILE = 5120;   // lcm(1024, 4 * R): 5 frames = 128 audio samples

int64_t gcd64(int64_t a, int64_t b)
{
    while (b) {
        const int64_t t = a % b;
        a = b;
        b = t;
    }
    return a;
}

std::mutex g_plan_mutex;
// (device, K, gain_db) -> plan; plans are tiny (a twiddle table) and live for the process
std::map<std::tuple<int, int, int>, b200_spectrum_plan*> g_plans;

b200_spectrum_plan* cached_plan(int K, int gain_db)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    // only the integer quotient gain_db / 10 reaches the arithmetic (cbb_main.c:112): one plan per decade,
    // so a client sweeping `spectrumgain` does not grow the cache
    gain_db = (gain_db / 10) * 10;
    auto key = std::make_tuple(dev, K, gain_db);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) return it->second;
    b200_spectrum_plan* pl = b200_spectrum_plan_create(CHAIN_N, CHAIN_N, K, 0, B200_WINDOW_RECT, gain_db);
    if (pl != nullptr) g_plans[key] = pl;
    return pl;
}

}  // namespace

extern "C" {

int64_t b200_chain_tile_samples(int R)
{
    if (R < 1 || R > 256) return B200_ERR_ARG;
    const int64_t a = CHAIN_N, b = 4 * (int64_t) R;
    return a / gcd64(a, b) * b;                 // lcm(1024, 4R): whole frames and whole audio samples (a multiple of 8)
}

int b200_chain_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int gain_db,
                    float* d_db, float* d_audio, int64_t audio_stride, uint8_t* d_avg_u8, int K_avg,
                    void* cuda_stream)
{
    return b200_chain_exec_r(d_iq, stream_stride_bytes, n_streams, n_samples, CHAIN_R, gain_db, d_db, d_audio,
                             audio_stride, d_avg_u8, K_avg, cuda_stream);
}

int b200_chain_exec_r(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                      int gain_db, float* d_db, float* d_audio, int64_t audio_stride, uint8_t* d_avg_u8, int K_avg,
                      void* cuda_stream)
{
    const int64_t tile = b200_chain_tile_samples(R);
    if (tile < 0) {
        set_error("chain exec: down factor %d outside [1, 256]", R);
        return B200_ERR_ARG;
    }
    if (d_iq == nullptr || n_streams < 0 || n_samples < 0 || n_samples % tile != 0) {
        set_error("chain exec: n_samples %lld must be a non-negative multiple of %lld", (long long) n_samples, (long long) tile);
        return B200_ERR_ARG;
    }
    if ((reinterpret_cast<uintptr_t>(d_iq) & 15) != 0 || (stream_stride_bytes & 15) != 0) {
        set_error("chain exec: IQ pointer and stream stride must be 16-byte aligned");
        return B200_ERR_ALIGN;
    }
    if (n_streams == 0 || n_samples == 0) return B200_OK;
    if (d_audio != nullptr && n_samples < fm_history_samples(R)) {
        // the carried state is the last 32 R input samples: a batch must hold at least that many
        set_error("chain exec: a batch of %lld samples is shorter than the FM history (%d samples at R = %d)",
                  (long long) n_samples, fm_history_samples(R), R);
        return B200_ERR_ARG;
    }
    if (d_avg_u8 != nullptr && (K_avg < 1 || (int64_t) K_avg * CHAIN_N > n_samples)) {     // before anything is launched
        set_error("chain exec: K_avg = %d does not fit the batch", K_avg);
        return B200_ERR_ARG;
    }
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    b200_spectrum_plan* pl = cached_plan(1, gain_db);
    if (pl == nullptr) return B200_ERR_CUDA;

    int rc;
    if (d_db != nullptr && d_audio != nullptr && R == CHAIN_R) {      // one pass over the IQ (chain_fused.cu)
        rc = launch_chain_fused(d_iq, stream_stride_bytes, n_streams, n_samples, spectrum_plan_db_offset(pl),
                                spectrum_plan_twiddle(pl), d_db, d_audio, audio_stride, stream);
        if (rc) return rc;
    } else {
        if (d_db != nullptr) {
            rc = b200_spectrum_exec(pl, d_iq, stream_stride_bytes, n_streams, n_samples / CHAIN_N, d_db, nullptr,
                                    nullptr, cuda_stream);
            if (rc) return rc;
        }
        if (d_audio != nullptr) {
            rc = b200_fm_exec(d_iq, stream_stride_bytes, n_streams, n_samples, R, d_audio, audio_stride, nullptr,
                              0, cuda_stream);
            if (rc) return rc;
        }
    }
    if (d_avg_u8 != nullptr) {
        b200_spectrum_plan* avg = cached_plan(K_avg, gain_db);
        if (avg == nullptr) return B200_ERR_CUDA;
        rc = b200_spectrum_exec(avg, d_iq, stream_stride_bytes, n_streams, 1, nullptr, nullptr, d_avg_u8, cuda_stream);
        if (rc) return rc;
    }
    return B200_OK;
}

}  // extern "C"

// ---- host-buffer session -----------------------------------------------------------------

struct b200_session {
    int n_streams = 0;
    int64_t max_samples = 0;
    int64_t tile = 0;                  // lcm(1024, 4R)
    IqRows rows;                       // [n_streams] [history | batch], the down factor R and the channel filter
    float* d_db = nullptr;             // [n_streams][max_samples]            (1024 bins per 1024 samples)
    float* d_audio = nullptr;          // [n_streams][max_samples / (4R)]
    uint8_t* d_avg = nullptr;          // [n_streams][1024] payload rows, allocated on first use (b200_session_products)
    int64_t position = 0;              // samples per stream consumed since create / reset (index of the next batch's first)
    uint32_t* d_phase_inc = nullptr;   // [n_streams][ch_cap], b200_session_channels, allocated on first use
    float* d_ch_audio = nullptr;       // [n_streams][ch_cap][max_samples / (4R)]
    int ch_cap = 0;                    // channels the two buffers above hold
    static constexpr int LANES = 4;
    cudaStream_t streams[LANES] = {};
    int device = 0;
};

// A batch every session call takes: n_samples in [0, max_samples] and whole tiles, and with a channel filter set,
// not shorter than its history (the carry copies the history from within the batch).
static int session_batch_check(const char* who, const b200_session* s, const uint8_t* h_iq, int64_t n_samples)
{
    if (s == nullptr || h_iq == nullptr || n_samples < 0 || n_samples > s->max_samples || n_samples % s->tile != 0) {
        set_error("%s: n_samples %lld must be a multiple of %lld and at most %lld", who, (long long) n_samples,
                  s ? (long long) s->tile : 0ll, s ? (long long) s->max_samples : 0ll);
        return B200_ERR_ARG;
    }
    if (n_samples > 0 && n_samples < s->rows.hist && s->rows.n_taps > 0) {
        set_error("%s: a batch of %lld samples is shorter than the channel filter's history (%d samples)", who,
                  (long long) n_samples, s->rows.hist);
        return B200_ERR_ARG;
    }
    return B200_OK;
}

// One batch of every stream, in groups of ceil(n_streams / 16) streams taken round-robin by the lanes, so that
// H2D copies, kernels and D2H copies of different groups overlap.  Per group: the 2-D copy of its IQ rows (iq_pitch
// bytes apart in h_iq) into the device rows, step(s0, ns, d_batch, lane) for its launches and copies back, and the
// history carry.
template <class Step>
static int session_groups(b200_session* s, const uint8_t* h_iq, int64_t iq_pitch, int64_t n_samples, Step step)
{
    const int lanes = b200_session::LANES;
    int group = (s->n_streams + 4 * lanes - 1) / (4 * lanes);
    if (group < 1) group = 1;
    int lane = 0;
    for (int s0 = 0; s0 < s->n_streams; s0 += group, lane = (lane + 1) % lanes) {
        const int ns = (s->n_streams - s0) < group ? (s->n_streams - s0) : group;
        cudaStream_t st = s->streams[lane];
        uint8_t* d_batch = s->rows.batch(s0);
        B200_CUDA_TRY(cudaMemcpy2DAsync(d_batch, (size_t) s->rows.pitch, h_iq + (size_t) s0 * (size_t) iq_pitch,
                                        (size_t) iq_pitch, (size_t) (2 * n_samples), (size_t) ns,
                                        cudaMemcpyHostToDevice, st));
        if (int rc = step(s0, ns, d_batch, st)) return rc;
        if (int rc = s->rows.carry(s0, ns, n_samples, st)) return rc;
    }
    return B200_OK;
}

namespace b200 {

// Submit one batch of every stream of the session without waiting: rows of the host arrays may be strided
// (pitches in bytes for h_iq, in floats for h_db / h_audio), which is how a multi-GPU host hands each device
// its streams s mod G of one global array.  d_avg_u8 (device, nullable): [n_streams][1024] payload rows.
int session_chain_submit(b200_session* s, const uint8_t* h_iq, int64_t iq_pitch_bytes, int64_t n_samples, int gain_db,
                         float* h_db, int64_t db_pitch, float* h_audio, int64_t audio_pitch, uint8_t* d_avg_u8, int K_avg)
{
    if (int rc = session_batch_check("session chain", s, h_iq, n_samples)) return rc;
    if (n_samples == 0) return B200_OK;
    const int64_t n_audio = n_samples / (4 * s->rows.R);
    const int rc = session_groups(s, h_iq, iq_pitch_bytes, n_samples, [&](int s0, int ns, uint8_t* d_batch, cudaStream_t st) {
        float* d_db = s->d_db + (size_t) s0 * (size_t) n_samples;
        float* d_audio = s->d_audio + (size_t) s0 * (size_t) n_audio;
        const int rc = b200_chain_exec_r(d_batch, s->rows.pitch, ns, n_samples, s->rows.R, gain_db, h_db ? d_db : nullptr,
                                         h_audio ? d_audio : nullptr, n_audio, d_avg_u8 ? d_avg_u8 + (size_t) s0 * 1024 : nullptr,
                                         K_avg, st);
        if (rc) return rc;
        if (h_db)
            B200_CUDA_TRY(cudaMemcpy2DAsync(h_db + (size_t) s0 * (size_t) db_pitch, sizeof(float) * (size_t) db_pitch, d_db,
                                            sizeof(float) * (size_t) n_samples, sizeof(float) * (size_t) n_samples,
                                            (size_t) ns, cudaMemcpyDeviceToHost, st));
        if (h_audio)
            B200_CUDA_TRY(cudaMemcpy2DAsync(h_audio + (size_t) s0 * (size_t) audio_pitch, sizeof(float) * (size_t) audio_pitch,
                                            d_audio, sizeof(float) * (size_t) n_audio, sizeof(float) * (size_t) n_audio,
                                            (size_t) ns, cudaMemcpyDeviceToHost, st));
        return B200_OK;
    });
    if (rc) return rc;
    s->position += n_samples;
    return B200_OK;
}

int session_wait(b200_session* s)
{
    for (int i = 0; i < b200_session::LANES; ++i) B200_CUDA_TRY(cudaStreamSynchronize(s->streams[i]));
    return B200_OK;
}

}  // namespace b200

extern "C" {

b200_session* b200_session_create(int n_streams, int64_t max_samples_per_batch)
{
    return b200_session_create_r(n_streams, max_samples_per_batch, CHAIN_R);
}

b200_session* b200_session_create_r(int n_streams, int64_t max_samples_per_batch, int R)
{
    const int64_t tile = b200_chain_tile_samples(R);
    if (tile < 0) {
        set_error("session: down factor %d outside [1, 256]", R);
        return nullptr;
    }
    if (n_streams < 1 || max_samples_per_batch < tile || max_samples_per_batch % tile != 0 ||
        max_samples_per_batch < fm_history_samples(R)) {
        set_error("session: max_samples_per_batch must be a positive multiple of %lld and at least %d", (long long) tile,
                  fm_history_samples(R));
        return nullptr;
    }
    b200_session* s = new b200_session();
    s->n_streams = n_streams;
    s->max_samples = max_samples_per_batch;
    s->tile = tile;
    bool ok = cudaGetDevice(&s->device) == cudaSuccess;
    ok = ok && cudaMalloc(&s->d_db, sizeof(float) * (size_t) n_streams * (size_t) max_samples_per_batch) == cudaSuccess;
    ok = ok && cudaMalloc(&s->d_audio, sizeof(float) * (size_t) n_streams * (size_t) (max_samples_per_batch / (4 * R))) ==
                   cudaSuccess;
    for (int i = 0; ok && i < b200_session::LANES; ++i)
        ok = cudaStreamCreateWithFlags(&s->streams[i], cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && s->rows.create(R, n_streams, max_samples_per_batch, s->streams[0]) == B200_OK;
    if (!ok) {
        set_error("session: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b200_session_destroy(s);
        return nullptr;
    }
    return s;
}

void b200_session_destroy(b200_session* s)
{
    if (s == nullptr) return;
    for (cudaStream_t st : s->streams)
        if (st) cudaStreamDestroy(st);
    s->rows.free();
    for (void* d : std::initializer_list<void*>{s->d_db, s->d_audio, s->d_avg, s->d_phase_inc, s->d_ch_audio})
        if (d != nullptr) cudaFree(d);
    delete s;
}

void b200_session_reset(b200_session* s)
{
    if (s == nullptr) return;
    s->rows.reset(s->streams[0]);
    s->position = 0;
}

int b200_session_channels(b200_session* s, const uint8_t* h_iq, int64_t n_samples, const uint32_t* h_phase_inc,
                          int n_channels, float* h_audio)
{
    if (s == nullptr || h_iq == nullptr || h_phase_inc == nullptr || h_audio == nullptr) {
        set_error("session channels: null argument");
        return B200_ERR_ARG;
    }
    if (n_channels < 1 || n_channels > B200_FM_MAX_CHANNELS) {
        set_error("session channels: n_channels %d outside [1, %d]", n_channels, B200_FM_MAX_CHANNELS);
        return B200_ERR_ARG;
    }
    if (int rc = session_batch_check("session channels", s, h_iq, n_samples)) return rc;
    if (n_samples == 0) return B200_OK;
    if (n_channels > s->ch_cap) {       // every earlier call has finished: the session calls wait for their work
        if (s->d_phase_inc) cudaFree(s->d_phase_inc);
        if (s->d_ch_audio) cudaFree(s->d_ch_audio);
        s->d_phase_inc = nullptr;
        s->d_ch_audio = nullptr;
        s->ch_cap = 0;
        const size_t rows = (size_t) s->n_streams * (size_t) n_channels;
        B200_CUDA_TRY(cudaMalloc((void**) &s->d_phase_inc, sizeof(uint32_t) * rows));
        B200_CUDA_TRY(cudaMalloc((void**) &s->d_ch_audio, sizeof(float) * rows * (size_t) (s->max_samples / (4 * s->rows.R))));
        s->ch_cap = n_channels;
    }
    const int64_t n_audio = n_samples / (4 * s->rows.R);
    const IqRows& r = s->rows;
    int rc = session_groups(s, h_iq, 2 * n_samples, n_samples, [&](int s0, int ns, uint8_t* d_batch, cudaStream_t st) {
        const size_t row0 = (size_t) s0 * (size_t) n_channels;
        const size_t rows = (size_t) ns * (size_t) n_channels;
        uint32_t* d_inc = s->d_phase_inc + row0;
        float* d_audio = s->d_ch_audio + row0 * (size_t) n_audio;
        B200_CUDA_TRY(cudaMemcpyAsync(d_inc, h_phase_inc + row0, sizeof(uint32_t) * rows, cudaMemcpyHostToDevice, st));
        const int rc = r.n_taps > 0
                           ? b200_fm_channels_exec_fir(d_batch, r.pitch, ns, n_samples, r.R, s->position, d_inc,
                                                       n_channels, d_audio, n_audio, nullptr, 0, r.d_taps, r.n_taps, st)
                           : b200_fm_channels_exec(d_batch, r.pitch, ns, n_samples, r.R, s->position, d_inc,
                                                   n_channels, d_audio, n_audio, nullptr, 0, st);
        if (rc) return rc;
        B200_CUDA_TRY(cudaMemcpyAsync(h_audio + row0 * (size_t) n_audio, d_audio, sizeof(float) * rows * (size_t) n_audio,
                                      cudaMemcpyDeviceToHost, st));
        return B200_OK;
    });
    if (rc) return rc;
    rc = b200::session_wait(s);
    if (rc) return rc;
    s->position += n_samples;
    return B200_OK;
}

int b200_session_set_channel_filter(b200_session* s, const float* h_taps, int n_taps)
{
    if (s == nullptr) {
        set_error("session channel filter: null session");
        return B200_ERR_ARG;
    }
    if (s->position != 0) {
        set_error("session channel filter: set it at stream position 0 (after create or b200_session_reset), "
                  "not at %lld", (long long) s->position);
        return B200_ERR_ARG;
    }
    // every earlier call has finished: the session calls wait for their work
    return s->rows.set_channel_filter("session channel filter", h_taps, n_taps, s->streams[0]);
}

int b200_session_chain(b200_session* s, const uint8_t* h_iq, int64_t n_samples, int gain_db, float* h_db,
                       float* h_audio)
{
    if (s == nullptr) {
        set_error("session chain: null session");
        return B200_ERR_ARG;
    }
    const int rc = b200::session_chain_submit(s, h_iq, 2 * n_samples, n_samples, gain_db, h_db, n_samples, h_audio,
                                              n_samples / (4 * s->rows.R), nullptr, 0);
    if (rc) return rc;
    return b200::session_wait(s);
}

int b200_session_products(b200_session* s, const uint8_t* h_iq, int64_t n_samples, int gain_db, int K_avg,
                          float* h_audio, uint8_t* h_avg_u8)
{
    if (s == nullptr || h_avg_u8 == nullptr || K_avg < 1) {
        set_error("session products: bad arguments");
        return B200_ERR_ARG;
    }
    if (s->d_avg == nullptr) B200_CUDA_TRY(cudaMalloc((void**) &s->d_avg, (size_t) s->n_streams * 1024));
    int rc = b200::session_chain_submit(s, h_iq, 2 * n_samples, n_samples, gain_db, nullptr, 0, h_audio,
                                        n_samples / (4 * s->rows.R), s->d_avg, K_avg);
    if (rc) return rc;
    rc = b200::session_wait(s);
    if (rc) return rc;
    B200_CUDA_TRY(cudaMemcpy(h_avg_u8, s->d_avg, (size_t) s->n_streams * 1024, cudaMemcpyDeviceToHost));
    return B200_OK;
}

}  // extern "C"

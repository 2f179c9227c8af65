// stream.cu -- b200_stream_*: the push-style entry point a signal_source callback calls
// (signal_source.h:7 `void (*)(const cmplx_u8*, int)`, fan-out at signal_source.c:29-35).
//
// Each of n independent dongle streams owns two pinned host slots of `batch_samples`
// (the "pinned host rings" of the north star).  b200_stream_push copies the callback's
// borrowed buffer (librtlsdr recycles it) into the current slot; a full slot is submitted
// without blocking: cudaMemcpyAsync to the stream's device row [history | batch], the fused
// chain kernel for that row, the history carry, and asynchronous copies of the dB rows and
// the audio back into pinned result buffers -- all on one of a small pool of CUDA streams,
// so batches of different dongles overlap.  Dongles that run in step (the usual case: same sample rate, same
// buffer size) fill their batches at the same time, so full slots are submitted in RUNS: when every stream
// of a group of up to 16 consecutive streams has its batch ready, the group goes out as one 2-D copy, one
// kernel launch over the group's rows and 2-D copies back -- seven CUDA calls per group instead of per stream.
// A stream that gets ahead of its group (its second slot fills) is submitted on its own, and poll / flush
// submit whatever is ready.  Results are handed to the caller's sinks from
// b200_stream_push / _poll / _flush on the calling thread (no hidden threads), in submission
// order per stream.  Re-blocking is aligned to stream start like rf_decimator.c:88-115, so
// results do not depend on how the source chunks the samples.
//
// FM channels (listeners at offsets inside a dongle's band): each stream has its own set of up to `chan_max`
// channels.  A batch takes the set that is current when its last sample is pushed (stored with the slot then), and a
// submitted run adds one launch of the runs-table channel kernel over its streams that have channels, after the
// chain kernel and before the history carry, and one 2-D copy back.
//
// Audio post-processing (b200_stream_set_audio_post, off by default): the centre audio of a run goes through
// b200_audio_post with one state row per dongle, and its channels through one b200_audio_post_rows call whose state
// rows belong to listener ids (stream_map_listeners).  The sinks then get the post-processed rows.
#include <string.h>

#include <vector>

#include "b200_common.cuh"

using namespace b200;

namespace {
constexpr int ST_R = 10;
constexpr int ST_SLOTS = 2;
constexpr int ST_LANES = 4;
constexpr int ST_GROUP = 16;       // streams submitted together when all of them are ready
}  // namespace

struct b200_stream {
    int n_streams = 0;
    int64_t batch = 0;                   // samples per batch (multiple of 5120)
    int gain_db = 0;
    IqRows rows;                         // [n_streams] [history | batch], the down factor R and the channel filter
    float* d_db = nullptr;               // [n_streams][batch]
    float* d_audio = nullptr;            // [n_streams][batch / (4R)]
    uint8_t* h_in = nullptr;             // pinned [n_streams][ST_SLOTS][2 * batch]
    float* h_db = nullptr;               // pinned [n_streams][ST_SLOTS][batch]
    float* h_audio = nullptr;            // pinned [n_streams][ST_SLOTS][batch / (4R)]
    uint8_t* d_payload = nullptr;        // [n_streams][1024]: K-frame averaged payload bytes of the batch start
    uint8_t* h_payload = nullptr;        // pinned [n_streams][ST_SLOTS][1024]
    int payload_K = 0;                   // 0 = no payload sink
    b200_payload_sink payload_sink = nullptr;
    cudaStream_t lanes[ST_LANES] = {};
    int chan_max = 0;                    // channel capacity per stream; 0 = no channel buffers yet
    b200_channel_audio_sink chan_sink = nullptr;
    float* d_chan = nullptr;             // [n_streams][chan_max][batch / (4R)]
    float* h_chan = nullptr;             // pinned [n_streams][ST_SLOTS][chan_max][batch / (4R)]
    struct ChannelSet {
        int n = 0;
        uint32_t inc[B200_FM_MAX_CHANNELS];
        int32_t id[B200_FM_MAX_CHANNELS];
    };
    struct PerStream {
        int64_t fill = 0;                // samples in the current slot
        int slot = 0;                    // slot being filled
        int64_t batches_submitted = 0;
        int64_t batches_delivered = 0;
        cudaEvent_t done[ST_SLOTS] = {};
        bool in_flight[ST_SLOTS] = {};
        bool ready[ST_SLOTS] = {};       // full, not yet submitted
        bool has_db[ST_SLOTS] = {};      // the submitted slot computed and copied per-frame dB rows
        ChannelSet channels;             // current listener set (b200_stream_set_channels)
        ChannelSet slot_channels[ST_SLOTS];     // the set of each full slot, taken when its last sample arrived
        bool has_chan[ST_SLOTS] = {};    // the submitted slot computed and copied channel audio
        // post-processing state slots of the listeners of the last submitted batch with channel work
        int64_t post_batch = -1;         // that batch's index; -1 = none
        bool slot_used[B200_FM_MAX_CHANNELS] = {};
        int32_t slot_id[B200_FM_MAX_CHANNELS];
    };
    std::vector<PerStream> st;
    int post_flags = 0;                  // b200_audio_post flags; 0 = raw audio
    double post_rate = 0.0;
    float* d_post_audio = nullptr;       // [n_streams][batch / (4R)]: post output, n_out floats a row
    float* d_post_state = nullptr;       // [n_streams][B200_AUDIO_POST_STATE_FLOATS]
    float* d_post_chan = nullptr;        // [n_streams][chan_max][batch / (4R)]: post output, n_out floats a row
    float* d_post_chan_state = nullptr;  // [n_streams][chan_max][B200_AUDIO_POST_STATE_FLOATS]: state slots
    int64_t n_audio() const { return batch / (4 * rows.R); }
    // audio samples a batch delivers per sink call
    int64_t n_out() const { return post_flags ? b200_audio_post_out_samples(n_audio(), post_flags) : n_audio(); }
    b200_spectrum_sink spectrum_sink = nullptr;
    b200_audio_sink audio_sink = nullptr;
    void* user = nullptr;
};

// A device buffer of `bytes` and its pinned host mirror of ST_SLOTS times that, or neither: on failure both are null
// and b200_last_error() says why, prefixed by `who`.
template <class T>
static bool alloc_slots(const char* who, T*& d, T*& h, size_t bytes)
{
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e == cudaSuccess) e = cudaHostAlloc(&h, ST_SLOTS * bytes, cudaHostAllocDefault);
    if (e == cudaSuccess) return true;
    set_error("%s: %s", who, cudaGetErrorString(e));
    if (d) cudaFree(d);
    d = nullptr;
    h = nullptr;
    return false;
}

static void stream_deliver(b200_stream* s, int i, bool block)
{
    b200_stream::PerStream& p = s->st[i];
    while (p.batches_delivered < p.batches_submitted) {
        const int slot = (int) (p.batches_delivered % ST_SLOTS);
        if (!p.in_flight[slot]) break;
        if (block) {
            if (cudaEventSynchronize(p.done[slot]) != cudaSuccess) break;
        } else if (cudaEventQuery(p.done[slot]) != cudaSuccess) {
            break;
        }
        const int64_t b = p.batches_delivered;
        const size_t off = ((size_t) i * ST_SLOTS + slot);
        if (s->payload_sink && s->payload_K > 0)
            s->payload_sink(s->user, i, b * (s->batch / 1024), s->payload_K, s->h_payload + off * 1024);
        // a sink installed after this batch was submitted without one gets nothing for it (there are no rows)
        if (s->spectrum_sink && p.has_db[slot])
            s->spectrum_sink(s->user, i, b * (s->batch / 1024), (int) (s->batch / 1024), s->h_db + off * (size_t) s->batch);
        const int64_t n_audio = s->n_audio();      // the host rows' pitch
        const int64_t n = s->n_out();
        if (s->audio_sink) s->audio_sink(s->user, i, b * n, (int) n, s->h_audio + off * (size_t) n_audio);
        if (s->chan_sink && p.has_chan[slot]) {
            const b200_stream::ChannelSet& cs = p.slot_channels[slot];
            for (int c = 0; c < cs.n; ++c)
                s->chan_sink(s->user, i, cs.id[c], b * n, (int) n,
                             s->h_chan + (off * (size_t) s->chan_max + (size_t) c) * (size_t) n_audio);
        }
        p.in_flight[slot] = false;
        ++p.batches_delivered;
    }
}

// The post-processing state slots of stream p's listeners cs in the batch being submitted (its batches_submitted-th),
// by id: a listener that was in the set of the stream's previous batch, when that batch had channel work, keeps its
// slot; any other takes a free slot and starts fresh.  Slots of listeners that left are free again.
static void stream_map_listeners(b200_stream::PerStream& p, const b200_stream::ChannelSet& cs, int* slot_of, bool* fresh)
{
    const bool carried = p.post_batch == p.batches_submitted - 1;
    bool used[B200_FM_MAX_CHANNELS] = {};
    for (int c = 0; c < cs.n; ++c) {
        slot_of[c] = -1;
        for (int k = 0; carried && k < B200_FM_MAX_CHANNELS; ++k)
            if (p.slot_used[k] && p.slot_id[k] == cs.id[c]) {
                slot_of[c] = k;
                used[k] = true;
                break;
            }
    }
    int k = 0;      // cs.n <= chan_max slots, so a listener without one finds a free one below chan_max
    for (int c = 0; c < cs.n; ++c) {
        fresh[c] = slot_of[c] < 0;
        if (fresh[c]) {
            while (used[k]) ++k;
            slot_of[c] = k;
            used[k] = true;
        }
        p.slot_id[slot_of[c]] = cs.id[c];
    }
    memcpy(p.slot_used, used, sizeof(used));
    p.post_batch = p.batches_submitted;
}

// Submit the ready slot `slot` of streams [a, b) as one unit.  All of them run on the lane of their group, so
// the batches of one stream stay ordered (the history carry of batch n precedes the copy of batch n + 1).
static int stream_submit_run(b200_stream* s, int a, int b, int slot)
{
    const int n = b - a;
    const size_t batch = (size_t) s->batch;
    const size_t n_audio = (size_t) s->n_audio();
    const size_t n_out = (size_t) s->n_out();
    const bool post = s->post_flags != 0;
    cudaStream_t lane = s->lanes[(a / ST_GROUP) % ST_LANES];
    const size_t off = (size_t) a * ST_SLOTS + (size_t) slot;            // first stream's slot; next stream: + ST_SLOTS
    uint8_t* d_batch = s->rows.batch(a);
    // per-frame dB rows exist only once a spectrum sink has been installed (b200_stream_set_sinks allocates them)
    const bool want_db = s->spectrum_sink != nullptr && s->d_db != nullptr && s->h_db != nullptr;
    float* d_db = want_db ? s->d_db + (size_t) a * batch : nullptr;
    float* d_audio = s->d_audio + (size_t) a * n_audio;
    uint8_t* d_pay = s->d_payload + (size_t) a * 1024;
    const bool want_payload = s->payload_sink != nullptr && s->payload_K > 0;
    B200_CUDA_TRY(cudaMemcpy2DAsync(d_batch, (size_t) s->rows.pitch, s->h_in + off * 2 * batch, ST_SLOTS * 2 * batch, 2 * batch,
                                    (size_t) n, cudaMemcpyHostToDevice, lane));
    // without a per-frame sink the dB rows are not computed at all: the FM kernel and the K-frame average only
    int rc = b200_chain_exec_r(d_batch, s->rows.pitch, n, s->batch, s->rows.R, s->gain_db, d_db, d_audio,
                               (int64_t) n_audio, want_payload ? d_pay : nullptr, want_payload ? s->payload_K : 0, lane);
    if (rc) return rc;
    // channels of the streams that have listeners: one runs-table launch over the group's rows
    const bool want_chan = s->chan_sink != nullptr && s->chan_max > 0;
    int chan_width = 0;
    if (want_chan) {
        b200_fm_channel_run runs[ST_GROUP];
        int n_runs = 0;
        b200_audio_post_row rows[ST_GROUP * B200_FM_MAX_CHANNELS];
        int n_rows = 0;
        for (int i = a; i < b; ++i) {
            const b200_stream::ChannelSet& cs = s->st[i].slot_channels[slot];
            if (post) {
                int slot_of[B200_FM_MAX_CHANNELS];
                bool fresh[B200_FM_MAX_CHANNELS];
                stream_map_listeners(s->st[i], cs, slot_of, fresh);
                for (int c = 0; c < cs.n; ++c)
                    rows[n_rows++] = {i * s->chan_max + c, i * s->chan_max + c, i * s->chan_max + slot_of[c], fresh[c]};
            }
            if (cs.n == 0) continue;
            b200_fm_channel_run& r = runs[n_runs++];
            r.stream = i - a;
            r.n_channels = cs.n;
            r.first_sample = s->st[i].batches_submitted * s->batch;
            r.audio_row = (int64_t) (i - a) * s->chan_max;
            memcpy(r.phase_inc, cs.inc, sizeof(uint32_t) * (size_t) cs.n);
            if (cs.n > chan_width) chan_width = cs.n;
        }
        if (n_runs > 0) {
            rc = launch_fm_channels_runs(d_batch, s->rows.pitch, n, s->batch, s->rows.R, runs, n_runs,
                                         s->d_chan + (size_t) a * (size_t) s->chan_max * n_audio, (int64_t) n_audio,
                                         (int64_t) n * s->chan_max, s->rows.d_taps, s->rows.n_taps, lane);
            if (rc) return rc;
        }
        if (n_rows > 0) {
            const int64_t n_chan_rows = (int64_t) s->n_streams * s->chan_max;
            rc = b200_audio_post_rows(s->d_chan, (int64_t) n_audio, n_chan_rows, (int64_t) n_audio, s->post_rate,
                                      s->post_flags, rows, n_rows, s->d_post_chan_state, n_chan_rows, s->d_post_chan,
                                      (int64_t) n_audio, n_chan_rows, lane);
            if (rc) return rc;
        }
    }
    if (post) {
        rc = b200_audio_post(d_audio, (int64_t) n_audio, n, (int64_t) n_audio, s->post_rate, s->post_flags,
                             s->d_post_state + (size_t) a * B200_AUDIO_POST_STATE_FLOATS,
                             s->d_post_audio + (size_t) a * n_audio, (int64_t) n_audio, lane);
        if (rc) return rc;
    }
    rc = s->rows.carry(a, n, s->batch, lane);
    if (rc) return rc;
    // the per-frame dB rows cross PCIe only if somebody listens (4 bytes per sample; the payload is 1 KB per batch)
    if (want_db)
        B200_CUDA_TRY(cudaMemcpy2DAsync(s->h_db + off * batch, ST_SLOTS * batch * sizeof(float), d_db, batch * sizeof(float),
                                        batch * sizeof(float), (size_t) n, cudaMemcpyDeviceToHost, lane));
    // post-processed rows hold n_out floats at the same pitch
    B200_CUDA_TRY(cudaMemcpy2DAsync(s->h_audio + off * n_audio, ST_SLOTS * n_audio * sizeof(float),
                                    post ? s->d_post_audio + (size_t) a * n_audio : d_audio, n_audio * sizeof(float),
                                    n_out * sizeof(float), (size_t) n, cudaMemcpyDeviceToHost, lane));
    if (want_payload)
        B200_CUDA_TRY(cudaMemcpy2DAsync(s->h_payload + off * 1024, ST_SLOTS * 1024, d_pay, 1024, 1024, (size_t) n,
                                        cudaMemcpyDeviceToHost, lane));
    // per stream, its first chan_width channel rows up to the last one's n_out floats (rows past a stream's own count
    // are not read on delivery)
    if (chan_width > 0) {
        const size_t block = (size_t) s->chan_max * n_audio * sizeof(float);
        B200_CUDA_TRY(cudaMemcpy2DAsync(s->h_chan + off * (size_t) s->chan_max * n_audio, ST_SLOTS * block,
                                        (post ? s->d_post_chan : s->d_chan) + (size_t) a * (size_t) s->chan_max * n_audio,
                                        block, ((size_t) (chan_width - 1) * n_audio + n_out) * sizeof(float), (size_t) n,
                                        cudaMemcpyDeviceToHost, lane));
    }
    for (int i = a; i < b; ++i) {
        b200_stream::PerStream& p = s->st[i];
        B200_CUDA_TRY(cudaEventRecord(p.done[slot], lane));
        p.ready[slot] = false;
        p.in_flight[slot] = true;
        p.has_db[slot] = want_db;
        p.has_chan[slot] = want_chan;
        ++p.batches_submitted;
    }
    return B200_OK;
}

// the slot stream i would submit next (its oldest full one), or -1
static int stream_ready_slot(const b200_stream* s, int i)
{
    const b200_stream::PerStream& p = s->st[i];
    const int slot = (int) (p.batches_submitted % ST_SLOTS);
    return p.ready[slot] ? slot : -1;
}

// submit the whole group of stream i if every member is ready with the same slot; returns 1 if it went out
static int stream_try_group(b200_stream* s, int i)
{
    const int a = (i / ST_GROUP) * ST_GROUP;
    const int b = a + ST_GROUP < s->n_streams ? a + ST_GROUP : s->n_streams;
    const int slot = stream_ready_slot(s, a);
    if (slot < 0) return 0;
    for (int k = a + 1; k < b; ++k)
        if (stream_ready_slot(s, k) != slot) return 0;
    const int rc = stream_submit_run(s, a, b, slot);
    return rc ? rc : 1;
}

// submit everything that is ready, in maximal runs of consecutive streams of one group with the same slot
static int stream_submit_ready(b200_stream* s)
{
    int i = 0;
    while (i < s->n_streams) {
        const int slot = stream_ready_slot(s, i);
        if (slot < 0) {
            ++i;
            continue;
        }
        const int group_end = (i / ST_GROUP + 1) * ST_GROUP < s->n_streams ? (i / ST_GROUP + 1) * ST_GROUP : s->n_streams;
        int j = i + 1;
        while (j < group_end && stream_ready_slot(s, j) == slot) ++j;
        const int rc = stream_submit_run(s, i, j, slot);
        if (rc) return rc;
        // the same stream may hold a second full slot: look at it again
    }
    return B200_OK;
}

// true once anything has been pushed: the settings that shape every batch are fixed from then on
static bool stream_started(const b200_stream* s)
{
    for (const auto& p : s->st)
        if (p.fill != 0 || p.batches_submitted != 0 || p.ready[0] || p.ready[1]) return true;
    return false;
}

// The post-processing buffers the stream lacks with post-processing `flags` and its channel capacity: the centre
// output and state rows (the state zeroed, waited for) and, with channels, their output rows and state slots (a slot
// is read only after a fresh start has written it).  On failure b200_last_error() says why.
static int stream_alloc_post(b200_stream* s, int flags)
{
    if (flags == 0) return B200_OK;
    const size_t ns = (size_t) s->n_streams, n_audio = (size_t) s->n_audio(), nc = (size_t) s->chan_max;
    const size_t state = sizeof(float) * B200_AUDIO_POST_STATE_FLOATS;
    if (s->d_post_audio == nullptr) B200_CUDA_TRY(cudaMalloc(&s->d_post_audio, sizeof(float) * ns * n_audio));
    if (s->d_post_state == nullptr) {
        B200_CUDA_TRY(cudaMalloc(&s->d_post_state, state * ns));
        B200_CUDA_TRY(cudaMemsetAsync(s->d_post_state, 0, state * ns, s->lanes[0]));
        B200_CUDA_TRY(cudaStreamSynchronize(s->lanes[0]));
    }
    if (nc > 0 && s->d_post_chan == nullptr) B200_CUDA_TRY(cudaMalloc(&s->d_post_chan, sizeof(float) * ns * nc * n_audio));
    if (nc > 0 && s->d_post_chan_state == nullptr) B200_CUDA_TRY(cudaMalloc(&s->d_post_chan_state, state * ns * nc));
    return B200_OK;
}

extern "C" {

b200_stream* b200_stream_create(int n_streams, int64_t batch_samples, int gain_db)
{
    return b200_stream_create_r(n_streams, batch_samples, gain_db, ST_R);
}

b200_stream* b200_stream_create_r(int n_streams, int64_t batch_samples, int gain_db, int R)
{
    const int64_t tile = b200_chain_tile_samples(R);
    if (tile < 0) {
        set_error("stream: down factor %d outside [1, 256]", R);
        return nullptr;
    }
    if (n_streams < 1 || batch_samples < tile || batch_samples % tile != 0 || batch_samples < fm_history_samples(R)) {
        // (the FM state is the last 32 R input samples: at R > 32 one tile is shorter than that)
        set_error("stream: batch_samples must be a positive multiple of %lld and at least %d", (long long) tile,
                  fm_history_samples(R));
        return nullptr;
    }
    b200_stream* s = new b200_stream();
    s->n_streams = n_streams;
    s->batch = batch_samples;
    s->gain_db = gain_db;
    const size_t ns = (size_t) n_streams;
    bool ok = alloc_slots("stream: allocation failed", s->d_audio, s->h_audio,
                          sizeof(float) * ns * (size_t) (batch_samples / (4 * R)));
    ok = ok && cudaHostAlloc(&s->h_in, ns * ST_SLOTS * 2 * (size_t) batch_samples, cudaHostAllocDefault) == cudaSuccess;
    ok = ok && alloc_slots("stream: allocation failed", s->d_payload, s->h_payload, ns * 1024);
    for (int i = 0; ok && i < ST_LANES; ++i) ok = cudaStreamCreateWithFlags(&s->lanes[i], cudaStreamNonBlocking) == cudaSuccess;
    s->st.resize(ns);
    for (auto& p : s->st)
        for (int k = 0; ok && k < ST_SLOTS; ++k) ok = cudaEventCreateWithFlags(&p.done[k], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && s->rows.create(R, n_streams, batch_samples, s->lanes[0]) == B200_OK;
    if (!ok) {
        set_error("stream: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b200_stream_destroy(s);
        return nullptr;
    }
    return s;
}

void b200_stream_destroy(b200_stream* s)
{
    if (s == nullptr) return;
    for (cudaStream_t lane : s->lanes)
        if (lane) {
            cudaStreamSynchronize(lane);
            cudaStreamDestroy(lane);
        }
    for (auto& p : s->st)
        for (cudaEvent_t ev : p.done)
            if (ev) cudaEventDestroy(ev);
    s->rows.free();
    for (void* d : std::initializer_list<void*>{s->d_db, s->d_audio, s->d_payload, s->d_chan, s->d_post_audio,
                                                s->d_post_state, s->d_post_chan, s->d_post_chan_state})
        if (d != nullptr) cudaFree(d);
    for (void* h : std::initializer_list<void*>{s->h_in, s->h_db, s->h_audio, s->h_payload, s->h_chan})
        if (h != nullptr) cudaFreeHost(h);
    delete s;
}

void b200_stream_set_sinks(b200_stream* s, b200_spectrum_sink spectrum_sink, b200_audio_sink audio_sink, void* user)
{
    if (s == nullptr) return;
    // The per-frame dB rows (4 bytes per sample on the device, twice that pinned on the host: 420 MB for 256 streams
    // of 204800 samples) exist only for callers that listen to them: allocated when the first spectrum sink arrives.
    if (spectrum_sink != nullptr && s->d_db == nullptr &&
        !alloc_slots("stream: dB row buffers", s->d_db, s->h_db, sizeof(float) * (size_t) s->n_streams * (size_t) s->batch))
        spectrum_sink = nullptr;      // reported through b200_last_error(); audio and payload keep working
    s->spectrum_sink = spectrum_sink;
    s->audio_sink = audio_sink;
    s->user = user;
}

int b200_stream_set_payload_sink(b200_stream* s, int K, b200_payload_sink sink)
{
    if (s == nullptr || K < 0 || (int64_t) K * 1024 > s->batch) {
        set_error("stream payload sink: K = %d frames do not fit a batch", K);
        return B200_ERR_ARG;
    }
    s->payload_K = sink ? K : 0;
    s->payload_sink = sink;
    return B200_OK;
}

int b200_stream_push(b200_stream* s, int stream, const uint8_t* samples, int len)
{
    if (s == nullptr || stream < 0 || stream >= s->n_streams || len < 0 || (len > 0 && samples == nullptr)) {
        set_error("stream push: bad arguments");
        return B200_ERR_ARG;
    }
    b200_stream::PerStream& p = s->st[stream];
    const uint8_t* src = samples;
    int64_t remaining = len;
    while (remaining > 0) {
        // the slot about to be written must be free: a batch still waiting for its group goes out on its own,
        // a batch in flight is waited for and delivered (two batches per stream at most)
        if (p.fill == 0 && p.ready[p.slot]) {
            const int rc = stream_submit_run(s, stream, stream + 1, p.slot);
            if (rc) return rc;
        }
        if (p.fill == 0 && p.in_flight[p.slot]) stream_deliver(s, stream, true);
        const int64_t room = s->batch - p.fill;
        const int64_t n = remaining < room ? remaining : room;
        uint8_t* dst = s->h_in + ((size_t) stream * ST_SLOTS + p.slot) * 2 * (size_t) s->batch + 2 * (size_t) p.fill;
        memcpy(dst, src, 2 * (size_t) n);
        src += 2 * n;
        p.fill += n;
        remaining -= n;
        if (p.fill == s->batch) {
            p.slot_channels[p.slot] = p.channels;      // the batch keeps the listener set of its last sample
            p.ready[p.slot] = true;
            p.slot = (p.slot + 1) % ST_SLOTS;
            p.fill = 0;
            const int rc = stream_try_group(s, stream);
            if (rc < 0) return rc;
        }
    }
    stream_deliver(s, stream, false);
    return B200_OK;
}

int b200_stream_poll(b200_stream* s)
{
    if (s == nullptr) return B200_ERR_ARG;
    if (int rc = stream_submit_ready(s)) return rc;         // batches waiting for a slower member of their group
    for (int i = 0; i < s->n_streams; ++i) stream_deliver(s, i, false);
    return B200_OK;
}

int b200_stream_flush(b200_stream* s)
{
    if (s == nullptr) return B200_ERR_ARG;
    if (int rc = stream_submit_ready(s)) return rc;
    for (int i = 0; i < s->n_streams; ++i) stream_deliver(s, i, true);
    return B200_OK;
}

int b200_stream_set_channel_sink(b200_stream* s, int max_channels, b200_channel_audio_sink sink)
{
    if (s == nullptr || max_channels < 1 || max_channels > B200_FM_MAX_CHANNELS ||
        (s->chan_max != 0 && max_channels != s->chan_max)) {
        set_error("stream channel sink: capacity %d must be in [1, %d] and stay what it was first (%d)", max_channels,
                  B200_FM_MAX_CHANNELS, s ? s->chan_max : 0);
        return B200_ERR_ARG;
    }
    if (s->chan_max == 0 && sink != nullptr) {      // the buffers come with the first sink, like the dB rows
        const size_t n_audio = (size_t) (s->batch / (4 * s->rows.R));
        if (!alloc_slots("stream channel sink: buffers", s->d_chan, s->h_chan,
                         sizeof(float) * (size_t) s->n_streams * (size_t) max_channels * n_audio))
            return B200_ERR_CUDA;
        s->chan_max = max_channels;
    }
    if (sink != nullptr)
        if (int rc = stream_alloc_post(s, s->post_flags)) return rc;
    s->chan_sink = sink;
    return B200_OK;
}

int b200_stream_set_channels(b200_stream* s, int stream, int n_channels, const uint32_t* h_phase_inc,
                             const int32_t* h_channel_ids)
{
    if (s == nullptr || stream < 0 || stream >= s->n_streams || s->chan_sink == nullptr || n_channels < 0 ||
        n_channels > s->chan_max || (n_channels > 0 && (h_phase_inc == nullptr || h_channel_ids == nullptr))) {
        set_error("stream channels: stream %d, %d channels (a channel sink of capacity %d is needed first)", stream,
                  n_channels, s ? s->chan_max : 0);
        return B200_ERR_ARG;
    }
    for (int c = 0; c < n_channels; ++c)
        for (int k = 0; k < c; ++k)
            if (h_channel_ids[k] == h_channel_ids[c]) {
                set_error("stream channels: channel id %d appears twice", (int) h_channel_ids[c]);
                return B200_ERR_ARG;
            }
    b200_stream::ChannelSet& cs = s->st[stream].channels;
    cs.n = n_channels;
    for (int c = 0; c < n_channels; ++c) {
        cs.inc[c] = h_phase_inc[c];
        cs.id[c] = h_channel_ids[c];
    }
    return B200_OK;
}

int b200_stream_set_channel_filter(b200_stream* s, const float* h_taps, int n_taps)
{
    if (s == nullptr) {
        set_error("stream channel filter: null stream");
        return B200_ERR_ARG;
    }
    if (stream_started(s)) {
        set_error("stream channel filter: set it before anything is pushed");
        return B200_ERR_ARG;
    }
    return s->rows.set_channel_filter("stream channel filter", h_taps, n_taps, s->lanes[0]);
}

int b200_stream_set_audio_post(b200_stream* s, int flags, double audio_rate_hz)
{
    if (s == nullptr || stream_started(s)) {
        set_error("stream audio post: set it before anything is pushed");
        return B200_ERR_ARG;
    }
    // a batch's audio is one call's n_audio: the resampler needs it a multiple of 16
    if (int rc = audio_post_check("stream audio post", flags, audio_rate_hz, s->n_audio(), nullptr, nullptr)) return rc;
    if (int rc = stream_alloc_post(s, flags)) return rc;
    s->post_flags = flags;
    s->post_rate = audio_rate_hz;
    return B200_OK;
}

int64_t b200_stream_pending_samples(const b200_stream* s, int stream)
{
    if (s == nullptr || stream < 0 || stream >= s->n_streams) return B200_ERR_ARG;
    return s->st[stream].fill;
}

}  // extern "C"

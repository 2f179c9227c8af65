// multi.cu -- multi-GPU through the C ABI: stream sharding and the one exchange of the path.
//
// Every piece of DSP state of the reference is per stream (rf_decimator.c:23,28; audio_main.c:77-79), so
// independent dongle streams shard across GPUs with no exchange on the data path: stream s lives on
// rank s mod G.  The only collective is at the end, when one consumer (the websocket server of main.c)
// wants the UI products of ALL streams -- the K-frame averaged u8 dB rows of cbb_main.c:121-130, 1 KB per
// stream: a gather to one rank.  NCCL carries it (grouped ncclSend / ncclRecv of each rank's contiguous
// rows, NVLink / NVSwitch underneath); a small kernel on the root then puts the rows into global stream
// order, reading the root's own rows straight from where the spectrum kernel wrote them.
//
// libnccl is loaded at run time (dlopen "libnccl.so.2"): a single-GPU host never needs it, and inside a
// process that already carries NCCL (torch.distributed) the same copy is reused.  Communicators are made
// either from a 128-byte id the host distributes itself (one process per GPU: b200_comm_unique_id on rank
// 0, b200_comm_create everywhere) or for all devices of one process (b200_comm_create_all).
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "b200_common.cuh"

using namespace b200;

namespace {

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int*) = nullptr;
};

std::mutex g_nccl_mutex;
NcclApi g_nccl;

const NcclApi* nccl()
{
    std::lock_guard<std::mutex> lock(g_nccl_mutex);
    if (g_nccl.handle != nullptr) return &g_nccl;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* n : names) {
        h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (h != nullptr) break;
    }
    if (h == nullptr) {
        set_error("multi-GPU: libnccl.so.2 not found (%s)", dlerror());
        return nullptr;
    }
    NcclApi a;
    a.handle = h;
#define B200_NCCL_SYM(field, name)                                  \
    *(void**) (&a.field) = dlsym(h, name);                          \
    if (a.field == nullptr) {                                       \
        set_error("multi-GPU: libnccl lacks %s", name);             \
        return nullptr;                                             \
    }
    B200_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    B200_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    B200_NCCL_SYM(CommInitAll, "ncclCommInitAll")
    B200_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    B200_NCCL_SYM(Send, "ncclSend")
    B200_NCCL_SYM(Recv, "ncclRecv")
    B200_NCCL_SYM(GroupStart, "ncclGroupStart")
    B200_NCCL_SYM(GroupEnd, "ncclGroupEnd")
    B200_NCCL_SYM(GetErrorString, "ncclGetErrorString")
    B200_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef B200_NCCL_SYM
    g_nccl = a;
    return &g_nccl;
}

#define B200_NCCL_TRY(api, expr)                                                                  \
    do {                                                                                          \
        ncclResult_t r__ = (expr);                                                                \
        if (r__ != ncclSuccess) {                                                                 \
            set_error("%s failed: %s (%s:%d)", #expr, (api)->GetErrorString(r__), __FILE__, __LINE__); \
            return B200_ERR_CUDA;                                                                 \
        }                                                                                         \
    } while (0)

// rows of rank r, local index i  ->  global row r + i * world.  `staged` holds the rows of every rank but
// `self` back to back in rank order; the root's own rows are read in place.
__global__ void gather_interleave_kernel(const uint32_t* __restrict__ staged, const uint32_t* __restrict__ own,
                                         uint32_t* __restrict__ out, int n_total, int world, int self, int row_words)
{
    const int g = blockIdx.x;                       // global row
    const int r = g % world;
    const int i = g / world;
    const uint32_t* src;
    if (r == self) {
        src = own + (size_t) i * row_words;
    } else {
        // rows before rank r in the staging buffer: sum over ranks q < r, q != self, of count(q)
        size_t before = 0;
        for (int q = 0; q < r; ++q)
            if (q != self) before += (size_t) ((n_total - q + world - 1) / world);
        src = staged + (before + (size_t) i) * row_words;
    }
    uint32_t* dst = out + (size_t) g * row_words;
    for (int w = threadIdx.x; w < row_words; w += blockDim.x) dst[w] = src[w];
}

}  // namespace

struct b200_comm {
    ncclComm_t comm;
    int world;
    int rank;
    int device;
    uint8_t* d_staging;
    size_t staging_bytes;
};

static int comm_reserve(b200_comm* c, size_t bytes)
{
    if (bytes <= c->staging_bytes) return B200_OK;
    if (c->d_staging) cudaFree(c->d_staging);
    c->d_staging = nullptr;
    c->staging_bytes = 0;
    B200_CUDA_TRY(cudaMalloc((void**) &c->d_staging, bytes));
    c->staging_bytes = bytes;
    return B200_OK;
}

static int shard_count(int n_streams, int world, int rank)
{
    return rank < n_streams ? (n_streams - rank + world - 1) / world : 0;
}

// the sends / receives of one rank (inside an open NCCL group)
static int gather_post(const NcclApi* api, b200_comm* c, const void* d_send, int n_total, int row_bytes, int root,
                       cudaStream_t stream)
{
    const int mine = shard_count(n_total, c->world, c->rank);
    if (c->rank != root) {
        if (mine > 0) B200_NCCL_TRY(api, api->Send(d_send, (size_t) mine * row_bytes, ncclUint8, root, c->comm, stream));
        return B200_OK;
    }
    size_t off = 0;
    for (int q = 0; q < c->world; ++q) {
        if (q == root) continue;
        const int cnt = shard_count(n_total, c->world, q);
        if (cnt > 0)
            B200_NCCL_TRY(api, api->Recv(c->d_staging + off, (size_t) cnt * row_bytes, ncclUint8, q, c->comm, stream));
        off += (size_t) cnt * row_bytes;
    }
    return B200_OK;
}

static int gather_finish(b200_comm* c, const void* d_send, int n_total, int row_bytes, void* d_recv, cudaStream_t stream)
{
    gather_interleave_kernel<<<n_total, 128, 0, stream>>>(reinterpret_cast<const uint32_t*>(c->d_staging),
                                                          reinterpret_cast<const uint32_t*>(d_send),
                                                          reinterpret_cast<uint32_t*>(d_recv), n_total, c->world, c->rank,
                                                          row_bytes / 4);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

static int gather_check_args(const b200_comm* c, const void* d_send, int n_total, int row_bytes, const void* d_recv, int root)
{
    if (c == nullptr || n_total < 0 || row_bytes <= 0 || row_bytes % 4 != 0 || root < 0 || root >= c->world) {
        set_error("gather rows: bad arguments (row_bytes must be a positive multiple of 4)");
        return B200_ERR_ARG;
    }
    if (shard_count(n_total, c->world, c->rank) > 0 && d_send == nullptr) {
        set_error("gather rows: rank %d has rows but no send buffer", c->rank);
        return B200_ERR_ARG;
    }
    if (c->rank == root && n_total > 0 && d_recv == nullptr) {
        set_error("gather rows: the root needs a receive buffer");
        return B200_ERR_ARG;
    }
    return B200_OK;
}

extern "C" {

int b200_shard_count(int n_streams, int world, int rank)
{
    if (n_streams < 0 || world < 1 || rank < 0 || rank >= world) return B200_ERR_ARG;
    return shard_count(n_streams, world, rank);
}

int b200_shard_stream(int n_streams, int world, int rank, int local_index)
{
    if (n_streams < 0 || world < 1 || rank < 0 || rank >= world || local_index < 0) return B200_ERR_ARG;
    const int g = rank + local_index * world;
    return g < n_streams ? g : B200_ERR_ARG;
}

int b200_comm_unique_id(uint8_t* id128)
{
    const NcclApi* api = nccl();
    if (api == nullptr || id128 == nullptr) return B200_ERR_CUDA;
    ncclUniqueId id;
    B200_NCCL_TRY(api, api->GetUniqueId(&id));
    static_assert(sizeof(id) == B200_COMM_ID_BYTES, "NCCL unique id size");
    memcpy(id128, &id, sizeof(id));
    return B200_OK;
}

b200_comm* b200_comm_create(const uint8_t* id128, int world, int rank)
{
    const NcclApi* api = nccl();
    if (api == nullptr) return nullptr;
    if (id128 == nullptr || world < 1 || rank < 0 || rank >= world) {
        set_error("comm create: bad arguments");
        return nullptr;
    }
    b200_comm* c = new b200_comm();
    memset(c, 0, sizeof(*c));
    c->world = world;
    c->rank = rank;
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclResult_t r = ncclSuccess;
    if (cudaGetDevice(&c->device) != cudaSuccess || (r = api->CommInitRank(&c->comm, world, id, rank)) != ncclSuccess) {
        set_error("comm create: %s", r != ncclSuccess ? api->GetErrorString(r) : cudaGetErrorString(cudaGetLastError()));
        delete c;
        return nullptr;
    }
    return c;
}

int b200_comm_create_all(int n_devices, b200_comm** comms)
{
    const NcclApi* api = nccl();
    if (api == nullptr) return B200_ERR_CUDA;
    if (n_devices < 1 || comms == nullptr) {
        set_error("comm create all: bad arguments");
        return B200_ERR_ARG;
    }
    std::vector<ncclComm_t> raw((size_t) n_devices);
    std::vector<int> devs((size_t) n_devices);
    for (int i = 0; i < n_devices; ++i) devs[i] = i;
    B200_NCCL_TRY(api, api->CommInitAll(raw.data(), n_devices, devs.data()));
    for (int i = 0; i < n_devices; ++i) {
        b200_comm* c = new b200_comm();
        memset(c, 0, sizeof(*c));
        c->comm = raw[i];
        c->world = n_devices;
        c->rank = i;
        c->device = i;
        comms[i] = c;
    }
    return B200_OK;
}

void b200_comm_destroy(b200_comm* c)
{
    if (c == nullptr) return;
    const NcclApi* api = nccl();
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(c->device);
    if (c->d_staging) cudaFree(c->d_staging);
    if (api != nullptr && c->comm != nullptr) api->CommDestroy(c->comm);
    cudaSetDevice(prev);
    delete c;
}

int b200_comm_world(const b200_comm* c) { return c ? c->world : B200_ERR_ARG; }
int b200_comm_rank(const b200_comm* c) { return c ? c->rank : B200_ERR_ARG; }

int b200_comm_nccl_version(void)
{
    const NcclApi* api = nccl();
    int v = 0;
    if (api == nullptr || api->GetVersion(&v) != ncclSuccess) return B200_ERR_CUDA;
    return v;
}

int b200_comm_gather_rows(b200_comm* c, const void* d_send, int n_streams_total, int row_bytes, void* d_recv, int root,
                          void* cuda_stream)
{
    if (int rc = gather_check_args(c, d_send, n_streams_total, row_bytes, d_recv, root)) return rc;
    const NcclApi* api = nccl();
    if (api == nullptr) return B200_ERR_CUDA;
    if (n_streams_total == 0) return B200_OK;
    cudaStream_t stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (c->rank == root) {
        const int others = n_streams_total - shard_count(n_streams_total, c->world, root);
        if (int rc = comm_reserve(c, (size_t) (others > 0 ? others : 1) * row_bytes)) return rc;
    }
    if (c->world > 1) {
        B200_NCCL_TRY(api, api->GroupStart());
        const int rc = gather_post(api, c, d_send, n_streams_total, row_bytes, root, stream);
        const ncclResult_t e = api->GroupEnd();
        if (rc) return rc;
        B200_NCCL_TRY(api, e);
    }
    if (c->rank == root) return gather_finish(c, d_send, n_streams_total, row_bytes, d_recv, stream);
    return B200_OK;
}

int b200_comm_gather_rows_all(b200_comm** comms, int n, const void* const* d_send, int n_streams_total, int row_bytes,
                              void* d_recv, int root, void* const* cuda_streams)
{
    if (comms == nullptr || d_send == nullptr || n < 1 || root < 0 || root >= n) {
        set_error("gather rows all: bad arguments");
        return B200_ERR_ARG;
    }
    const NcclApi* api = nccl();
    if (api == nullptr) return B200_ERR_CUDA;
    for (int i = 0; i < n; ++i)
        if (int rc = gather_check_args(comms[i], d_send[i], n_streams_total, row_bytes, i == root ? d_recv : nullptr, root)) return rc;
    if (n_streams_total == 0) return B200_OK;
    int prev = 0;
    B200_CUDA_TRY(cudaGetDevice(&prev));
    B200_CUDA_TRY(cudaSetDevice(comms[root]->device));
    const int others = n_streams_total - shard_count(n_streams_total, n, root);
    if (int rc = comm_reserve(comms[root], (size_t) (others > 0 ? others : 1) * row_bytes)) return rc;
    int rc = B200_OK;
    if (n > 1) {
        B200_NCCL_TRY(api, api->GroupStart());
        for (int i = 0; i < n && rc == B200_OK; ++i) {
            cudaSetDevice(comms[i]->device);
            rc = gather_post(api, comms[i], d_send[i], n_streams_total, row_bytes, root,
                             reinterpret_cast<cudaStream_t>(cuda_streams ? cuda_streams[i] : nullptr));
        }
        const ncclResult_t e = api->GroupEnd();
        if (rc == B200_OK && e != ncclSuccess) {
            set_error("ncclGroupEnd failed: %s", api->GetErrorString(e));
            rc = B200_ERR_CUDA;
        }
    }
    if (rc == B200_OK) {
        cudaSetDevice(comms[root]->device);
        rc = gather_finish(comms[root], d_send[root], n_streams_total, row_bytes, d_recv,
                           reinterpret_cast<cudaStream_t>(cuda_streams ? cuda_streams[root] : nullptr));
    }
    cudaSetDevice(prev);
    return rc;
}

}  // extern "C"

// ---- one process, G GPUs, host buffers: b200_multi ------------------------------------------------
//
// The host-buffer session of chain.cu, once per device, behind one object: stream s of the caller's global
// arrays goes to device s mod G (rows of the host arrays are simply read and written with a pitch of G
// rows, no repacking), every device runs the chain on its own streams concurrently, and the per-stream
// payload rows are gathered on device 0 by b200_comm_gather_rows_all before they go back to the host.

struct b200_multi {
    int G;
    int n_streams;
    int64_t max_samples;
    int gain_db;
    int K_avg;
    std::vector<b200_session*> sess;       // per device, n_local streams (null if the device has none)
    std::vector<b200_comm*> comms;
    std::vector<uint8_t*> d_avg;           // per device: [n_local][1024]
    uint8_t* d_all;                        // device 0: [n_streams][1024] in global stream order
};

extern "C" {

void b200_multi_destroy(b200_multi* m)
{
    if (m == nullptr) return;
    int prev = 0;
    cudaGetDevice(&prev);
    for (int g = 0; g < m->G; ++g) {
        cudaSetDevice(g);
        if (g < (int) m->sess.size() && m->sess[g]) b200_session_destroy(m->sess[g]);
        if (g < (int) m->d_avg.size() && m->d_avg[g]) cudaFree(m->d_avg[g]);
        if (g == 0 && m->d_all) cudaFree(m->d_all);
    }
    for (b200_comm* c : m->comms)
        if (c) b200_comm_destroy(c);
    cudaSetDevice(prev);
    delete m;
}

b200_multi* b200_multi_create(int n_gpus, int n_streams, int64_t max_samples_per_batch, int gain_db, int K_avg)
{
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess || n_gpus < 1 || n_gpus > have) {
        set_error("multi: %d GPUs asked for, %d visible", n_gpus, have);
        return nullptr;
    }
    if (n_streams < 1 || K_avg < 0 || (int64_t) K_avg * 1024 > max_samples_per_batch) {
        set_error("multi: bad arguments");
        return nullptr;
    }
    int prev = 0;
    cudaGetDevice(&prev);
    b200_multi* m = new b200_multi();
    m->G = n_gpus;
    m->n_streams = n_streams;
    m->max_samples = max_samples_per_batch;
    m->gain_db = gain_db;
    m->K_avg = K_avg;
    m->d_all = nullptr;
    m->sess.assign((size_t) n_gpus, nullptr);
    m->d_avg.assign((size_t) n_gpus, nullptr);
    m->comms.assign((size_t) n_gpus, nullptr);
    bool ok = true;
    for (int g = 0; g < n_gpus && ok; ++g) {
        const int n_local = shard_count(n_streams, n_gpus, g);
        ok = cudaSetDevice(g) == cudaSuccess;
        if (ok && n_local > 0) {
            m->sess[g] = b200_session_create(n_local, max_samples_per_batch);
            ok = m->sess[g] != nullptr && cudaMalloc((void**) &m->d_avg[g], (size_t) n_local * 1024) == cudaSuccess;
        }
        if (ok && g == 0) ok = cudaMalloc((void**) &m->d_all, (size_t) n_streams * 1024) == cudaSuccess;
    }
    if (ok && K_avg > 0 && n_gpus > 1) ok = b200_comm_create_all(n_gpus, m->comms.data()) == B200_OK;
    cudaSetDevice(prev);
    if (!ok) {
        if (b200_last_error()[0] == 0) set_error("multi: allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        b200_multi_destroy(m);
        return nullptr;
    }
    return m;
}

int b200_multi_chain(b200_multi* m, const uint8_t* h_iq, int64_t n_samples, float* h_db, float* h_audio, uint8_t* h_avg_u8)
{
    if (m == nullptr || h_iq == nullptr || (h_avg_u8 != nullptr && m->K_avg < 1)) {
        set_error("multi chain: bad arguments (payload rows need K_avg >= 1 at create)");
        return B200_ERR_ARG;
    }
    int prev = 0;
    B200_CUDA_TRY(cudaGetDevice(&prev));
    const int G = m->G;
    const int64_t n_audio = n_samples / 40;
    int rc = B200_OK;
    for (int g = 0; g < G && rc == B200_OK; ++g) {          // every device gets its streams s mod G; nothing waits yet
        if (m->sess[g] == nullptr) continue;
        cudaSetDevice(g);
        rc = session_chain_submit(m->sess[g], h_iq + (size_t) g * 2 * (size_t) n_samples, (int64_t) G * 2 * n_samples, n_samples,
                                  m->gain_db, h_db ? h_db + (size_t) g * (size_t) n_samples : nullptr, (int64_t) G * n_samples,
                                  h_audio ? h_audio + (size_t) g * (size_t) n_audio : nullptr, (int64_t) G * n_audio,
                                  h_avg_u8 ? m->d_avg[g] : nullptr, m->K_avg);
    }
    for (int g = 0; g < G; ++g) {
        if (m->sess[g] == nullptr) continue;
        cudaSetDevice(g);
        const int rw = session_wait(m->sess[g]);
        if (rc == B200_OK) rc = rw;
    }
    if (rc == B200_OK && h_avg_u8 != nullptr) {
        cudaSetDevice(0);
        if (G > 1) {
            std::vector<const void*> sends((size_t) G);
            for (int g = 0; g < G; ++g) sends[g] = m->d_avg[g];
            rc = b200_comm_gather_rows_all(m->comms.data(), G, sends.data(), m->n_streams, 1024, m->d_all, 0, nullptr);
        } else if (cudaMemcpy(m->d_all, m->d_avg[0], (size_t) m->n_streams * 1024, cudaMemcpyDeviceToDevice) != cudaSuccess) {
            rc = B200_ERR_CUDA;
        }
        if (rc == B200_OK) {
            cudaSetDevice(0);
            if (cudaMemcpy(h_avg_u8, m->d_all, (size_t) m->n_streams * 1024, cudaMemcpyDeviceToHost) != cudaSuccess) {
                set_error("multi chain: %s", cudaGetErrorString(cudaGetLastError()));
                rc = B200_ERR_CUDA;
            }
        }
    }
    cudaSetDevice(prev);
    return rc;
}

}  // extern "C"

// b200_common.cuh -- shared device helpers (sm_100a): mbarrier + 1-D bulk TMA copies, tensor
// memory, error plumbing, and the one declaration of each internal host launcher and helper.
// No CPU fallback anywhere: a failed CUDA call surfaces as B200_ERR_CUDA.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/b200sdr.h"

namespace b200 {

// ---- host-side error plumbing ---------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
int sm_count();

#define B200_CUDA_TRY(expr)                                                              \
    do {                                                                                 \
        cudaError_t e__ = (expr);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            ::b200::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),  \
                              __FILE__, __LINE__);                                       \
            return B200_ERR_CUDA;                                                        \
        }                                                                                \
    } while (0)

// Opt a kernel into more than 48 KB of dynamic shared memory, once per (kernel, device): the
// attribute belongs to the device's copy of the function, and a process may drive several GPUs.
int ensure_dynamic_smem(const void* kernel, int bytes);
// Resident CTAs per SM for (kernel, block, smem), cached per device like the attribute.
int cached_occupancy(const void* kernel, int block_threads, int smem_bytes);

#define B200_LAUNCH_CHECK()                                                              \
    do {                                                                                 \
        ::b200::g_launches.fetch_add(1, std::memory_order_relaxed);                      \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) {                                                        \
            ::b200::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                              __FILE__, __LINE__);                                       \
            return B200_ERR_CUDA;                                                        \
        }                                                                                \
    } while (0)

// ---- host-side launchers and helpers, each implemented next to its kernels ---------------
struct SpecParams;
struct Spec64kExtra;
struct FmParams;

// The spectrum launchers get at least one row, and an N that b200_spectrum_plan_create accepted: capi.cu checks the rest.
int launch_spectrum1024(const SpecParams& p, cudaStream_t stream);
int launch_spectrum2048(const SpecParams& p, cudaStream_t stream);
int launch_spectrum4096(const SpecParams& p, cudaStream_t stream);
int launch_spectrum_mx1024(const SpecParams& p, cudaStream_t stream);
int launch_spectrum64k(const SpecParams& p, const Spec64kExtra& x, int N, cudaStream_t stream);
int launch_spectrum_generic(const SpecParams& p, int N, int kind, float2* scratch, float* acc_scratch, int scratch_ctas,
                            cudaStream_t stream);
int spectrum_generic_scratch_ctas();
// the two fields of the (capi.cu-private) plan layout the fused chain launch needs
const float2* spectrum_plan_twiddle(const b200_spectrum_plan* plan);
float spectrum_plan_db_offset(const b200_spectrum_plan* plan);
int launch_chain_fused(const uint8_t* d_iq, int64_t stride, int n_streams, int64_t n_samples, float db_offset,
                       const float2* twiddle, float* d_db, float* d_audio, int64_t audio_stride, cudaStream_t stream);

int launch_fm_chain(const FmParams& p, cudaStream_t stream);
int fm_history_samples(int R);
int launch_iq_history_carry(uint8_t* iq, int64_t stride, int n_streams, int64_t n_samples, int hist_samples,
                            cudaStream_t stream);
int launch_iq_history_reset(uint8_t* iq, int64_t stride, int n_streams, int hist_samples, cudaStream_t stream);

// FM channels: taps NULL with T = 0 is the boxcar, else T in [1, B200_FM_MAX_CHANNEL_TAPS] device taps
int launch_fm_channels(const uint8_t* iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                       int64_t first_sample, const uint32_t* phase_inc, int n_channels, float* audio,
                       int64_t audio_stride, float* baseband, int64_t baseband_stride, const float* taps, int T,
                       cudaStream_t stream);
int launch_fm_channels_runs(const uint8_t* iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                            const b200_fm_channel_run* runs, int n_runs, float* audio, int64_t audio_stride,
                            int64_t n_audio_rows, const float* taps, int T, cudaStream_t stream);
int fm_channels_fir_history_samples(int R, int T);
int fm_channel_filter_design(int R, int T, double cutoff_hz, double atten_db, double fs, float* h);

// audio_post.cu: the flag, rate and length rules of b200_audio_post, b200_audio_post_rows and
// b200_stream_set_audio_post (B200_ERR_ARG, b200_last_error() prefixed by `who`); alpha and runin are nullable
int audio_post_check(const char* who, int flags, double audio_rate_hz, int64_t n_audio, float* alpha, int* runin);

// The device IQ rows of a session or a push stream: one row per stream, [history | batch], the history being the
// last `hist` samples of the stream's previous batch (128 before the first).  The history is the FM chain's 32 R,
// or the longer one the channel filter reaches back over.  Each call that launches work does it on `stream`.
struct IqRows {
    int R = 0;                     // down factor of the FM branch
    int n_rows = 0;
    int64_t max_batch = 0;         // samples
    int hist = 0;                  // samples
    int64_t pitch = 0;             // bytes per row: 2 * (hist + max_batch)
    uint8_t* d_base = nullptr;     // [n_rows][pitch]
    float* d_taps = nullptr;       // the channel filter's n_taps taps, nullptr = the boxcar
    int n_taps = 0;

    // rows with a 32 R history, reset and waited for; on failure free() releases what was allocated
    int create(int R, int n_rows, int64_t max_batch, cudaStream_t stream);
    void free();
    uint8_t* batch(int i) const { return d_base + (int64_t) i * pitch + 2 * (int64_t) hist; }
    // every row's history back to 128, waited for
    int reset(cudaStream_t stream);
    // the history of rows [i0, i0 + n) <- the last `hist` samples of their batch of n_samples
    int carry(int i0, int n, int64_t n_samples, cudaStream_t stream);
    // At stream position 0, with every earlier call on the rows finished: n_taps host taps (0 = the boxcar) become
    // the filter, and when it needs another history, new rows with it, reset, replace the old ones.  Waits on
    // `stream`.  On failure nothing changes.
    int set_channel_filter(const char* who, const float* h_taps, int n_taps, cudaStream_t stream);

private:
    int alloc(int hist_samples, cudaStream_t stream);
};

// chain.cu: one batch of a host-buffer session, submitted without waiting (multi.cu drives one session per device)
int session_chain_submit(b200_session* s, const uint8_t* h_iq, int64_t iq_pitch_bytes, int64_t n_samples, int gain_db,
                         float* h_db, int64_t db_pitch, float* h_audio, int64_t audio_pitch, uint8_t* d_avg_u8, int K_avg);
int session_wait(b200_session* s);

// ---- device: mbarrier + bulk async copy (TMA, 1-D) -------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
    return (uint32_t) __cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make mbarrier initialisation visible to the async proxy before the first TMA uses it
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// order this thread's prior generic-proxy smem accesses before later async-proxy ones
__device__ __forceinline__ void fence_proxy_async_smem()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}

// global -> shared bulk copy through the TMA unit (SASS: UBLKCP); completion is signalled
// on `bar` as `bytes` transaction bytes.  dst, src 16-byte aligned, bytes % 16 == 0.
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- device: tensor memory (tcgen05, one CTA) -------------------------------------------
// A TMEM address is lane << 16 | column.  A warp may only touch the 32 lanes of its quadrant, lanes
// 32 (warp % 4) .. 32 (warp % 4) + 31; in the 32x32b shape thread t of the warp reads or writes lane
// 32 (warp % 4) + t, 16 consecutive 32-bit columns from the address's column on (.x16).

// Whole warp: allocate n_cols columns (a power of two, 32..512) of every lane; the base address lands in *slot.
// Publish it to the other warps with tmem_fence_before_sync, a block barrier and tmem_fence_after_sync.
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t n_cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)),
                 "r"(n_cols)
                 : "memory");
}

// Whole warp: free what tmem_alloc returned.  Every allocation must be freed before the CTA exits.
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t n_cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(n_cols) : "memory");
}

// Whole warp: this CTA allocates no more, so a CTA waiting for tensor memory on this SM need not wait for it.
__device__ __forceinline__ void tmem_relinquish_alloc_permit()
{
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

// Whole warp: r[] -> 16 columns of this thread's lane.  Complete only after tmem_wait_st.
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
                 "%13, %14, %15, %16};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                 "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                 : "memory");
}

// Whole warp: 16 columns of this thread's lane -> r[].  The load is asynchronous: r[] may be read only after
// tmem_wait_ld(r), which also keeps the compiler from moving a use of r[] above the wait.
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, "
                 "%13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
}

// Whole warp: wait until every tcgen05.ld this thread issued has landed; r[] is the destination of the last one.
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&r)[16])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}

// Whole warp: wait until every tcgen05.st this thread issued has been written.
__device__ __forceinline__ void tmem_wait_st()
{
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Order this thread's tcgen05 operations before (after) a thread synchronisation that follows (precedes) it.
__device__ __forceinline__ void tmem_fence_before_sync()
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_fence_after_sync()
{
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// drop a 128-byte line from L2 without writing it back (its contents are dead)
__device__ __forceinline__ void l2_discard_128(const void* ptr)
{
    asm volatile("discard.global.L2 [%0], 128;" ::"l"(ptr) : "memory");
}

// log2 on the MUFU unit, flush-to-zero form: no denormal pre-scaling instructions.  Inputs
// here are sums of squares of integers (exact zero or >= 1), never denormal.  lg2(0) = -inf.
__device__ __forceinline__ float lg2_ftz(float x)
{
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

#endif  // __CUDACC__

}  // namespace b200

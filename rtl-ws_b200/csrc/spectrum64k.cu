// spectrum64k.cu -- 65536-point power spectra (BASELINE config 4: wideband spectrogram,
// Hann window, 50 % overlap), one CTA per frame, four-step through an L2-resident scratch
// (sm_100a).  The same kernel, with R = N / 1024 polyphase branches as a template parameter, serves N = 16384
// (R = 16) and 32768 (R = 32), which no other kernel of the library covers (the generic kernel ran them below
// 100 Gsamples/s).  The description below is for R = 64.
//
// 65536 = 64 x 1024, decimation in time by 64:
//   X[k + 1024 q] = sum_{r<64} W_64^(r q) * ( W_N^(r k) * F_r[k] ),   F_r = FFT_1024( x[64 m + r] ).
// A CTA (8 warps, one per SM) owns one frame at a time:
//   0. the 128 KB of IQ bytes are copied into shared memory with 128-bit loads; every 128-byte
//      row (one m, all 64 r) is word-swizzled by (m mod 32) so that the stride-128-byte reads
//      of a polyphase branch hit 32 different banks;
//   1. warp w runs the 32x32 register transform (fft1024_warp.cuh) on branches r = w, w+8, ...,
//      multiplies by W_N^(r k) (table stored [r][k], read coalesced) and writes Z[r][k] to this
//      CTA's 512 KB slice of a global scratch meant to stay in the 126 MB L2 (ncu: most of it does
//      not -- see DESIGN.md section 4.6);
//   2. block barrier; thread t takes k = t, t+256, ... (< 1024): 64 coalesced loads of Z[.][k],
//      a 64-point FFT in registers, |X|^2, K-frame accumulation with the cumulative
//      DC-position patch (spectrum.c:30-33), dB / power / u8, coalesced stores.
// Arithmetic per frame as in spectrum1024.cu (spectrum.c:15-58, cbb_main.c:112-128); the window
// (an extension; the reference is rectangular; periodic Hann is the only one the plan offers) is
// computed, not tabulated.
#include "b200_common.cuh"
#include "fft1024_warp.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

constexpr int S64_THREADS = 256;
constexpr int S64_WARPS = 8;                                              // R branches and 1024 columns divide evenly
constexpr int s64_smem(int R) { return 2 * 1024 * R + S64_WARPS * FFT1024_XCH_BYTES + 16; }

// R-point in-register transform of phase 2 (input in bit-reversed order, output natural)
template <int R>
__device__ __forceinline__ void fft_columns(c64 (&z)[R])
{
    if constexpr (R == 64) {
        fft_dit64(z);
    } else if constexpr (R == 32) {
        float2 unused[32];
        fft_dit32<false>(z, unused);
    } else {
        fft_dit_small<R>(z);
    }
}

template <int R, bool WINDOW, bool MULTI>
__global__ void __launch_bounds__(S64_THREADS, 1) spectrum64k_kernel(const SpecParams p, const Spec64kExtra x)
{
    constexpr int N64K = 1024 * R;                      // the frame length of this instantiation (65536 for R = 64)
    constexpr int S64_FRAME_BYTES = 2 * N64K;
    constexpr int WPR = R / 2;                          // 32-bit words per row (one m, all R branches)
    constexpr int RP = 32 / WPR;                        // rows per 128 bytes
    extern __shared__ __align__(128) uint8_t smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    uint32_t* frame32 = reinterpret_cast<uint32_t*>(smem);                 // [1024 rows][WPR words], swizzled
    float2* xch = reinterpret_cast<float2*>(smem + S64_FRAME_BYTES + warp * FFT1024_XCH_BYTES);
    float* dc_slot = reinterpret_cast<float*>(smem + S64_FRAME_BYTES + S64_WARPS * FFT1024_XCH_BYTES);

    c64* Z = reinterpret_cast<c64*>(x.scratch) + (size_t) blockIdx.x * N64K;     // [64][1024]
    float* acc = x.acc + (size_t) blockIdx.x * N64K;                              // [65536], MULTI only

    const int64_t total = (int64_t) p.n_streams * p.n_rows;
    const int K = MULTI ? p.K : 1;
    const float dboff = p.db_offset - 16.0f * DB_PER_LOG2;

    auto emit = [&](size_t row_base, int bin, float pw) {
        const int col = (bin + N64K / 2) & (N64K - 1);
        const float db = fmaf(DB_PER_LOG2, lg2_ftz(pw), dboff);
        if (p.db) __stcs(p.db + row_base + col, db);
        if (p.power) __stcs(p.power + row_base + col, pw * FFT1024_POWER_SCALE);
        if (p.db_u8) {
            int m = __float2int_rz(db);
            m = m < 0 ? 0 : (m > 255 ? 255 : m);
            p.db_u8[row_base + col] = (uint8_t) m;
        }
    };

    // A CTA takes a CONTIGUOUS range of (stream, row) items, so that with 50 % overlap (hop = N/2, the
    // spectrogram of BASELINE config 4) consecutive frames share half their samples and only the new half is
    // fetched: logical row m of the frame lives in physical row m ^ flip, flip alternating between 0 and 512
    // (the swizzle depends on m mod 32 only, which the flip leaves alone).
    const int64_t per_cta = (total + gridDim.x - 1) / gridDim.x;
    const int64_t item_begin = (int64_t) blockIdx.x * per_cta;
    const int64_t item_end = item_begin + per_cta < total ? item_begin + per_cta : total;
    int flip = 0;

    // frames in the order this CTA transforms them: seq = (item - item_begin) * K + j
    const int64_t n_seq = item_begin < item_end ? (item_end - item_begin) * K : 0;
    auto frame_of = [&](int64_t seq) {
        const int64_t item = item_begin + seq / K;
        const int j = (int) (seq - (seq / K) * K);
        const int64_t s = item / p.n_rows;
        const int64_t row = item - s * p.n_rows;
        return p.iq + s * p.stream_stride_bytes + 2 * (row * p.row_hop + (int64_t) j * p.hop);
    };
    // 0. frame -> shared memory with 4-byte cp.async copies (LDGSTS: no registers, nothing waits).  A row (one m,
    //    all R branches) is WPR words; word w of logical row m lands in word w ^ ((m / RP) % WPR) of physical row
    //    m ^ flip_, so that the stride-(2R)-byte reads of a branch hit 32 different banks (RP rows share 128 bytes).
    //    Thread t copies words t + 256 i.  The fetch of frame seq + 1 is issued as soon as phase 1 of frame seq is over
    //    (its bytes are dead then) and lands while phase 2 runs.
    auto fetch = [&](const uint8_t* frame, int flip_, bool half) {
        const uint32_t dst0 = smem_u32(frame32);
        const uint8_t* src0 = frame + 4 * tid;
#pragma unroll 8
        for (int i = half ? R : 0; i < 2 * R; ++i) {
            const int W = tid + S64_THREADS * i;
            const int m = W / WPR, w = W % WPR;
            const uint32_t dst = dst0 + (uint32_t) (((m ^ flip_) * WPR + (w ^ ((m / RP) % WPR))) * 4);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src0 + 4 * S64_THREADS * i) : "memory");
        }
    };
    if (n_seq > 0) fetch(frame_of(0), 0, false);
    const uint8_t* resident = n_seq > 0 ? frame_of(0) : nullptr;      // global address of the frame in shared memory

    for (int64_t item = item_begin; item < item_end; ++item) {
        const size_t row_base = (size_t) item * N64K;
        float dcacc = 0.0f;

        for (int j = 0; j < K; ++j) {
            const int64_t seq = (item - item_begin) * K + j;
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncthreads();          // the frame is in shared memory; Z and dc_slot of the previous frame are free

            // ---- 1. polyphase branches r = warp, warp + 8, ...  (the lane-private inter-pass twiddles
            //         are re-read per frame so that they are not live during phase 2) ----
            float2 tw[32];
            fft1024_load_twiddles(p.twiddle, lane, tw);
            for (int r = warp; r < R; r += S64_WARPS) {
                c64 a[32];
                // Hann window of sample R*(32*n1 + lane) + r without a table:
                //   w = 1/2 - 1/2 cos(2 pi n1 / 32 + phi),  phi = 2 pi (R lane + r) / N
                // (the [r][m] window table cost 256 KB of L2 reads per frame per SM)
                float cphi = 1.0f, sphi = 0.0f;
                if (WINDOW) sincospif((float) (R * lane + r) * (2.0f / (float) N64K), &sphi, &cphi);
                {
                    const c64 bias1 = cpack(8421376.0f, 8421376.0f);        // 2^23 + 256 * 128
                    // rows m < 512 (n1 < 16) and m >= 512 sit in the halves chosen by `flip`: two base pointers,
                    // every load still base + compile-time offset; m = 32 n1 + lane, so the swizzle is per lane
                    const int sw = (lane / RP) % WPR;
                    const int col = (((r >> 1) ^ sw) << 2) + ((r & 1) << 1);
                    const uint8_t* fb_lo = reinterpret_cast<const uint8_t*>(frame32) + flip * (2 * R) + lane * (2 * R) + col;
                    const uint8_t* fb_hi = reinterpret_cast<const uint8_t*>(frame32) - flip * (2 * R) + lane * (2 * R) + col;
#pragma unroll
                    for (int n1 = 0; n1 < 32; ++n1) {
                        const uint8_t* fb = n1 < 16 ? fb_lo : fb_hi;
                        const uint32_t v = *reinterpret_cast<const uint16_t*>(fb + 32 * n1 * (2 * R));
                        const int q = bitrev<32>(n1);
                        a[q] = cpack(__uint_as_float(__byte_perm(v, 0x4B000000u, 0x7504)),
                                     __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7514)));
                        if (WINDOW) {
                            const float w = fmaf(0.5f * sin32(n1), sphi, fmaf(-0.5f * cos32(n1), cphi, 0.5f));
                            a[q] = cmul2(csub(a[q], bias1), cpack(w, w));
                        }
                    }
                }
                c64 b[32];
                fft1024_transform<!WINDOW>(a, tw, xch, lane, b);
                const float2* twr = x.twiddle_rk + r * 1024;
                c64* zr = Z + r * 1024;
#pragma unroll
                for (int k2 = 0; k2 < 32; ++k2) {
                    const int k = lane + 32 * k2;
                    c64 z = b[k2];
                    if (r > 0) {
                        const float2 w = __ldg(&twr[k]);
                        z = cmul(z, w.x, w.y);
                    }
                    zr[k] = z;
                }
            }
            __syncthreads();          // Z[.][.] of this frame is complete and visible to the CTA
            if (seq + 1 < n_seq) {
                const uint8_t* next = frame_of(seq + 1);
                const bool half = (next == resident + S64_FRAME_BYTES / 2);   // the old second half is the new first half
                flip = half ? flip ^ 512 : 0;
                resident = next;
                fetch(next, flip, half);
            }

            // ---- 2. R-point transforms across r for k = tid + 256 g ----
            for (int g = 0; g < (1024 + S64_THREADS - 1) / S64_THREADS; ++g) {
                const int k = tid + S64_THREADS * g;
                if (k >= 1024) break;
                c64 z[R];
#pragma unroll
                for (int r = 0; r < R; ++r) z[bitrev<R>(r)] = Z[r * 1024 + k];
                fft_columns<R>(z);
#pragma unroll
                for (int q = 0; q < R; ++q) {
                    float re, im;
                    cunpack(z[q], re, im);
                    const float pw = fmaf(re, re, im * im);
                    const int bin = k + 1024 * q;
                    if (MULTI) {
                        acc[bin] = (j == 0 ? 0.0f : acc[bin]) + pw;
                    } else if (bin != 0) {
                        emit(row_base, bin, pw);
                    }
                    if (k == 1023 && q == R - 1) dcacc = fmaf((float) (K - j), pw, dcacc);  // bin N-1
                }
            }
            if (j == K - 1 && tid == 1023 % S64_THREADS) *dc_slot = dcacc;
            __syncthreads();          // frame32 / Z are rewritten by the next frame; dc_slot is visible
            // Z(frame) is dead now.  Its 4096 dirty L2 lines would otherwise be written back to HBM before the
            // next frame overwrites them (the reuse distance across 148 CTAs is ~200 MB, more than the L2 holds:
            // ncu showed 6 of the 8 GB of scratch writes per 524 M samples going to DRAM): drop them instead.
#pragma unroll 4
            for (int i = tid; i < N64K * 8 / 128; i += S64_THREADS)
                l2_discard_128(reinterpret_cast<const char*>(Z) + 128 * (size_t) i);
        }

        // spectrum.c:30-33: the DC position takes the (cumulative) value of its left neighbour, bin N-1
        if (!MULTI) {
            if (tid == 0) emit(row_base, 0, *dc_slot);
        } else {
            const float dc = *dc_slot;
            for (int bin = tid; bin < N64K; bin += S64_THREADS) emit(row_base, bin, bin == 0 ? dc : acc[bin]);
        }
        __syncthreads();
    }
}

// Tried and dropped (round 2, measured): asking the L2 to keep the Z scratch -- an access-policy window with the
// persisting property over the 74 MB, backed by a set-aside of the same size.  DRAM writes went UP (6.9 -> 11.9 GB per
// 524 M samples: what is left of the L2 no longer absorbs the streaming rows) and the kernel lost 3 % (123 -> 119
// Gsamples/s).  A sweep of the set-aside (32 / 64 / 79 MB = the device's maximum, misses left at normal priority) gave
// 7.6 / 11.9 / 11.9 GB of DRAM writes against 7.0 without it: no size helps.  A four-CTA cluster kernel that keeps Z in
// distributed shared memory removes the scratch altogether, but measured slower (DESIGN.md 4.6).
template <int R>
static int launch_scratch(const SpecParams& p, const Spec64kExtra& x, cudaStream_t stream)
{
    const int64_t total = (int64_t) p.n_streams * p.n_rows;
    auto kern = p.K > 1 ? (p.window ? spectrum64k_kernel<R, true, true> : spectrum64k_kernel<R, false, true>)
                        : (p.window ? spectrum64k_kernel<R, true, false> : spectrum64k_kernel<R, false, false>);
    if (int rc = ensure_dynamic_smem((const void*) kern, s64_smem(R))) return rc;
    int64_t grid = x.scratch_ctas;
    if (grid > total) grid = total;
    kern<<<(unsigned) grid, S64_THREADS, s64_smem(R), stream>>>(p, x);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace

// N = 65536 (and, through the same kernel, 16384 and 32768): x.scratch holds [scratch_ctas][N] complex, x.twiddle_rk
// [N / 1024][1024], x.acc [scratch_ctas][N] floats when K > 1
int launch_spectrum64k(const SpecParams& p, const Spec64kExtra& x, int N, cudaStream_t stream)
{
    return N == 65536 ? launch_scratch<64>(p, x, stream)
                      : (N == 32768 ? launch_scratch<32>(p, x, stream) : launch_scratch<16>(p, x, stream));
}

}  // namespace b200

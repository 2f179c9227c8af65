// spectrum_generic.cu -- power spectra for any power-of-two N (16 <= N <= 65536) and any of
// the reference's three input types, one CTA per output row (sm_100a).
//
// This is the general-shape kernel behind the compat entry points
// (spectrum_add_cmplx_s32 / spectrum_add_real_f32, spectrum.c:65-99, which have no callers
// in the reference) and behind frame lengths that have no specialised kernel.  The
// reference's default shape (N = 1024, u8 IQ) runs in spectrum1024.cu instead.
//
// Stockham autosort radix-4 passes (one radix-2 clean-up when log2 N is odd); the two
// ping-pong buffers live in shared memory up to N = 8192 and in an L2-resident global
// scratch above that.  Arithmetic per frame follows spectrum.c:15-35 exactly as in the
// specialised kernel: unpack, forward DFT, fftshift, |X|^2 accumulate over K frames with the
// cumulative DC-position patch, then the dB epilogue of cbb_main.c:125-128.
#include "b200_common.cuh"
#include "spectrum_kernels.cuh"

namespace b200 {

namespace {

enum InputKind { IN_CU8 = 0, IN_CS32 = 1, IN_RF32 = 2 };

__device__ __forceinline__ float2 cmul(float2 a, float2 w)
{
    return make_float2(fmaf(-a.y, w.y, a.x * w.x), fmaf(a.x, w.y, a.y * w.x));
}

constexpr int GEN_THREADS = 512;
constexpr int GEN_SMEM_MAX_N = 8192;

template <int KIND>
__device__ __forceinline__ float2 load_sample(const void* frame, int i)
{
    if (KIND == IN_CU8) {
        // spectrum.c:56-57; the /128 is applied to the power (2^-14), which is exact
        const uint16_t v = reinterpret_cast<const uint16_t*>(frame)[i];
        return make_float2((float) ((int) (v & 0xff) - 128), (float) ((int) (v >> 8) - 128));
    } else if (KIND == IN_CS32) {
        // spectrum.c:74-75
        const int2 v = reinterpret_cast<const int2*>(frame)[i];
        return make_float2((float) v.x, (float) v.y);
    } else {
        // spectrum.c:92-93 (no /128 on this path: undo the common 2^-14 power scale with *128)
        return make_float2(reinterpret_cast<const float*>(frame)[i] * 128.0f, 0.0f);
    }
}

template <int KIND>
__global__ void __launch_bounds__(GEN_THREADS) spectrum_generic_kernel(const SpecParams p, const int N,
                                                                       const int sample_bytes, float2* scratch,
                                                                       float* acc_scratch)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float2* buf0;
    float2* buf1;
    float* acc;
    if (N <= GEN_SMEM_MAX_N) {
        buf0 = reinterpret_cast<float2*>(smem_raw);
        buf1 = buf0 + N;
        acc = reinterpret_cast<float*>(buf1 + N);
    } else {
        buf0 = scratch + (size_t) blockIdx.x * 2 * N;
        buf1 = buf0 + N;
        acc = acc_scratch + (size_t) blockIdx.x * N;
    }
    const int tid = threadIdx.x;
    const int64_t total = (int64_t) p.n_streams * p.n_rows;
    const int half = N / 2;

    for (int64_t item = blockIdx.x; item < total; item += gridDim.x) {
        const int64_t s = item / p.n_rows;
        const int64_t r = item - s * p.n_rows;
        for (int i = tid; i < N; i += GEN_THREADS) acc[i] = 0.0f;
        float dcacc = 0.0f;     // meaningful in the thread that owns bin N-1

        for (int j = 0; j < p.K; ++j) {
            const uint8_t* frame = p.iq + s * p.stream_stride_bytes +
                                   (r * p.row_hop + (int64_t) j * p.hop) * sample_bytes;
            for (int i = tid; i < N; i += GEN_THREADS) {
                float2 v = load_sample<KIND>(frame, i);
                if (p.window != nullptr) {
                    const float w = p.window[i];
                    v.x *= w;
                    v.y *= w;
                }
                buf0[i] = v;
            }
            __syncthreads();

            float2* x = buf0;
            float2* y = buf1;
            int n = N;
            int st = 1;
            while (n >= 4) {
                const int n1 = n >> 2;
                const int tstep = N / n;
                for (int t = tid; t < (N >> 2); t += GEN_THREADS) {
                    const int pp = t / st;
                    const int q = t - pp * st;
                    const float2 a = x[q + st * pp];
                    const float2 b = x[q + st * (pp + n1)];
                    const float2 c = x[q + st * (pp + 2 * n1)];
                    const float2 d = x[q + st * (pp + 3 * n1)];
                    const float2 apc = make_float2(a.x + c.x, a.y + c.y);
                    const float2 amc = make_float2(a.x - c.x, a.y - c.y);
                    const float2 bpd = make_float2(b.x + d.x, b.y + d.y);
                    const float2 jbmd = make_float2(-(b.y - d.y), b.x - d.x);      // i * (b - d)
                    const float2 w1 = __ldg(&p.twiddle[(pp * tstep) & (N - 1)]);
                    const float2 w2 = __ldg(&p.twiddle[(2 * pp * tstep) & (N - 1)]);
                    const float2 w3 = __ldg(&p.twiddle[(3 * pp * tstep) & (N - 1)]);
                    y[q + st * (4 * pp + 0)] = make_float2(apc.x + bpd.x, apc.y + bpd.y);
                    y[q + st * (4 * pp + 1)] = cmul(make_float2(amc.x - jbmd.x, amc.y - jbmd.y), w1);
                    y[q + st * (4 * pp + 2)] = cmul(make_float2(apc.x - bpd.x, apc.y - bpd.y), w2);
                    y[q + st * (4 * pp + 3)] = cmul(make_float2(amc.x + jbmd.x, amc.y + jbmd.y), w3);
                }
                __syncthreads();
                float2* tmp = x; x = y; y = tmp;
                n >>= 2;
                st <<= 2;
            }
            if (n == 2) {
                for (int q = tid; q < st; q += GEN_THREADS) {
                    const float2 a = x[q];
                    const float2 b = x[q + st];
                    y[q] = make_float2(a.x + b.x, a.y + b.y);
                    y[q + st] = make_float2(a.x - b.x, a.y - b.y);
                }
                __syncthreads();
                float2* tmp = x; x = y; y = tmp;
            }

            // spectrum.c:23-34, display order
            for (int i = tid; i < N; i += GEN_THREADS) {
                const int bin = (i + half) & (N - 1);
                const float2 v = x[bin];
                const float pw = fmaf(v.x, v.x, v.y * v.y);
                acc[i] += pw;
                if (i == half - 1) dcacc = fmaf((float) (p.K - j), pw, dcacc);
            }
            __syncthreads();
        }

        // the thread that owns display index N/2-1 also owns ... not necessarily N/2: go through acc[]
        if (((half - 1) % GEN_THREADS) == tid) acc[half] = dcacc;
        __syncthreads();
        const size_t row = (size_t) item * N;
        for (int i = tid; i < N; i += GEN_THREADS) {
            const float pw = acc[i];
            const float db = fmaf(3.01029995663981195f, __log2f(pw), p.db_offset);
            if (p.db) p.db[row + i] = db;
            if (p.power) p.power[row + i] = pw * (1.0f / 16384.0f);
            if (p.db_u8) {
                int m = __float2int_rz(db);
                m = m < 0 ? 0 : (m > 255 ? 255 : m);
                p.db_u8[row + i] = (uint8_t) m;
            }
        }
        __syncthreads();
    }
}

}  // namespace

// CTAs the N > 8192 form runs (and the number of per-CTA work arrays the caller must provide)
int spectrum_generic_scratch_ctas()
{
    return sm_count() * 2;
}

// kind: 0 = cmplx_u8, 1 = cmplx_s32, 2 = real f32.  N > 8192 works out of global memory: `scratch` is
// [scratch_ctas][2][N] complex and `acc_scratch` [scratch_ctas][N], owned by the caller's plan (one exec at a time).
int launch_spectrum_generic(const SpecParams& p, int N, int kind, float2* scratch, float* acc_scratch, int scratch_ctas,
                            cudaStream_t stream)
{
    const int64_t total = (int64_t) p.n_streams * p.n_rows;
    const int sample_bytes = kind == IN_CU8 ? 2 : (kind == IN_CS32 ? 8 : 4);
    int grid;
    int smem = 0;
    if (N <= GEN_SMEM_MAX_N) {
        smem = 2 * N * 8 + N * 4;
        const int per_sm = smem > 113 * 1024 ? 1 : (smem > 56 * 1024 ? 2 : 3);
        grid = sm_count() * per_sm;
        scratch = nullptr;
        acc_scratch = nullptr;
    } else {
        if (scratch == nullptr || acc_scratch == nullptr || scratch_ctas <= 0) {
            set_error("spectrum: N = %d needs the plan's scratch", N);
            return B200_ERR_ARG;
        }
        grid = scratch_ctas;
    }
    if (grid > total) grid = (int) total;
    auto kern = kind == IN_CU8 ? spectrum_generic_kernel<IN_CU8>
                               : (kind == IN_CS32 ? spectrum_generic_kernel<IN_CS32> : spectrum_generic_kernel<IN_RF32>);
    if (smem > 48 * 1024)
        if (int rc = ensure_dynamic_smem((const void*) kern, smem)) return rc;
    kern<<<grid, GEN_THREADS, smem, stream>>>(p, N, sample_bytes, scratch, acc_scratch);
    B200_LAUNCH_CHECK();
    return B200_OK;
}

}  // namespace b200

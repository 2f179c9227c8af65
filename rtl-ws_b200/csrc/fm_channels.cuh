// fm_channels.cuh -- what the boxcar channel kernel (fm_channels.cu) and the FIR channel kernel (fm_channels_fir.cu)
// share: the tile geometry, the parameter block, the exact-phase rotation and the byte unpacking.
#pragma once

#include "b200_common.cuh"
#include "fft_regs.cuh"

namespace b200 {

constexpr int FC_T = 62;                    // audio samples per tile
constexpr int FC_ND = 4 * FC_T + 32;        // 280 decimated samples, local index 0 <-> 4*n0 - 32
constexpr int FC_NW = 2 * FC_T + 10;        // 134 first-stage outputs
constexpr int FC_WARPS = 9;                 // 9 * 31 = 279 demodulator outputs = local indices 1..279
constexpr int FC_THREADS = FC_WARPS * 32;
constexpr int FC_DEMOD = 288;               // floats per channel (8-byte aligned rows)
constexpr int FC_WORK = 144;

struct FcParams {
    const uint8_t* iq;              // stream 0, first sample of the batch (history lies before it)
    int64_t stream_stride_bytes;
    int n_streams;
    int64_t n_samples;
    int R;
    int64_t first_sample;           // absolute index of the batch's first sample, a multiple of 4R
    const uint32_t* phase_inc;      // [n_streams][n_channels]
    int n_channels;
    float* audio;                   // row s * n_channels + c
    int64_t audio_stride;           // floats
    float2* baseband;               // nullable, row s * n_channels + c
    int64_t baseband_stride;        // complex samples
};

// A b200_fm_channel_run as the kernels read it: the launcher computes the first decimated sample first_sample / R
// (mod 2^32, like every phase) once on the host, so that no tile divides a 64-bit position.
struct FcRun {
    int32_t stream;
    int32_t n_channels;
    uint32_t first_dec;
    int64_t audio_row;
    uint32_t phase_inc[B200_FM_MAX_CHANNELS];
};

// The runs form (b200_fm_channels_exec_runs): tile t belongs to run t / tiles_per_stream, and each run names its own
// IQ row, channel count, increments, stream position and audio row.  The base's n_streams is the number of runs; its
// first_sample, phase_inc, n_channels and baseband are unused.  Passed by value as a __grid_constant__ parameter
// (~9.8 KB): per-run fields are read from the constant bank, and nothing is copied to the device.
struct FcRunsParams : FcParams {
    FcRun runs[B200_FM_MAX_RUNS];
};

// exp(-j theta) for theta = 2 pi phi / 2^32, phi read as int32 so theta is in [-pi, pi).  MUFU sin / cos: the
// argument carries <= 3.1e-7 rad of rounding (int -> float and the product), sin.approx / cos.approx <= 5.1e-7 on
// [-pi, pi]: <= 8.2e-7 absolute per component.  phi = 0 is exactly (1, 0).
__device__ __forceinline__ void rotation(uint32_t phi, float& c, float& s)
{
    const float x = (float) (int32_t) phi * 1.46291807926715968e-9f;      // pi / 2^31
    __sincosf(x, &s, &c);
    if (phi == 0u) {
        c = 1.0f;
        s = 0.0f;
    }
}

// byte `sel` of v minus 128 as a float, both halves of a packed pair: 0x4B0000bb is the float 2^23 + b
__device__ __forceinline__ c64 byte_pair(uint32_t v, uint32_t sel)
{
    const float u = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7540u | sel));
    return cadd(cpack(u, u), cpack(-8388736.0f, -8388736.0f));
}

// the run of tile group q in the runs form (FcRunsParams / FirRunsParams); nullptr in the uniform form
template <bool RUNS, class P>
__device__ __forceinline__ const FcRun* fc_run(const P& p, int q)
{
    if constexpr (RUNS) return &p.runs[q];
    else return nullptr;
}

// host side: the FIR launchers (fm_channels_fir.cu), called by launch_fm_channels / launch_fm_channels_runs after
// their checks; T in [1, B200_FM_MAX_CHANNEL_TAPS]
int launch_fm_channels_fir(const FcParams& p, int64_t tiles_per_stream, const float* taps, int T, cudaStream_t stream);
int launch_fm_channels_fir_runs(const FcRunsParams& p, int64_t tiles_per_stream, const float* taps, int T,
                                int max_channels, cudaStream_t stream);

}  // namespace b200

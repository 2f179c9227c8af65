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

}  // namespace b200

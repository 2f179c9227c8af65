// spectrum_kernels.cuh -- parameter block shared by the spectrum kernels and their launcher.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

struct SpecParams {
    const uint8_t* iq;            // stream 0, sample 0 (cmplx_u8 wire layout)
    int64_t stream_stride_bytes;  // between streams
    int n_streams;
    int64_t n_rows;               // output rows per stream
    int hop;                      // samples between the K frames of one row
    int K;                        // frames accumulated per row
    int64_t row_hop;              // samples between rows
    float* db;                    // [n_streams][n_rows][N] or null
    float* power;                 // [n_streams][n_rows][N] or null
    uint8_t* db_u8;               // [n_streams][n_rows][N] or null
    float db_offset;              // 10*log10(g / (K * 2^14)): folds gain, /count and the 1/128 input scale
    const float2* twiddle;        // exp(-2*pi*i*k/N), k = 0..N-1 (device); the 1024-point table for u8 input at
                                  // N = 8192 and the four-step sizes (16384..65536)
    const float2* twiddle_n;      // u8 input from N = 2048 up: the inter-pass table W_N^(r c), [N/64][64] below N = 8192,
                                  // else [N/1024][1024] (the four-step kernel reads it as Spec64kExtra::twiddle_rk); else null
    const float* window;          // N floats (device) or null = rectangular
};

// extra tables / scratch of the 65536-point four-step kernel (spectrum64k.cu)
struct Spec64kExtra {
    float2* scratch;              // [scratch_ctas][64][1024] complex: Z[r][k], L2-resident
    float* acc;                   // [scratch_ctas][65536] power accumulators (K > 1), else null
    const float2* twiddle_rk;     // [64][1024]: exp(-2*pi*i*r*k/65536)
    int scratch_ctas;
};

}  // namespace b200

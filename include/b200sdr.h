/*
 * b200sdr.h -- C ABI of libb200sdr.so: the B200-native (sm_100a) IQ processing path for
 * rtl-ws.  Plain C, plain pointers and sizes; no CUDA or torch types appear in any
 * signature (a CUDA stream is passed as an opaque `void*`, NULL = the default stream).
 *
 * Two layers are exported:
 *
 *   1. The reference's own DSP interface, symbol for symbol (include/rtlws_compat.h):
 *      spectrum_*, rf_decimator_*, cic_decimate, halfband_decimate.  An unmodified
 *      cbb_main.c / audio_main.c / main.c links against this library instead of the
 *      reference's spectrum.o / rf_decimator.o / resample.o.
 *
 *   2. The batched / streaming extension declared here (SURVEY.md section 8b "required
 *      extension"), which is what carries throughput: many frames and many independent
 *      dongle streams per launch, device-resident or fed from pinned host rings.
 *
 * Every entry point names the reference code whose arithmetic it reproduces
 * (paths relative to the reference's src/).  Results match that code bit-for-bit for
 * integer stages and within the tolerances of BASELINE.json for floating point.
 * There is no CPU fallback: without a usable CUDA device every call fails with
 * B200_ERR_CUDA and b200_last_error() says why.
 */
#ifndef B200SDR_H
#define B200SDR_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_ARG (-1)     /* size / parameter mismatch (the reference's -1) */
#define B200_ERR_OVERRUN (-2) /* internal overrun (the reference's -2) */
#define B200_ERR_CUDA (-3)    /* CUDA runtime failure or no device; see b200_last_error() */
#define B200_ERR_ALIGN (-4)   /* pointer / stride / hop not aligned as documented */

/* ---- library ------------------------------------------------------------------------ */

/* Selects the CUDA device for the calling thread and warms the context.  Optional: every
 * other call initialises lazily on the current device. */
int b200_init(int device);
/* Last error text of the calling thread ("" if none). */
const char* b200_last_error(void);
/* Number of kernel launches issued by this library since load (all threads). */
uint64_t b200_launch_count(void);
/* SM count of the current device (grid sizing is a multiple of it). */
int b200_sm_count(void);

/* ---- batched power spectrum ------------------------------------------------------------
 *
 * Replaces, for many frames at once:
 *   spectrum.c:47-58   u8 -> ((x - 128) / 128) unpack           (+ optional window, extension)
 *   spectrum.c:21      fftw_execute: unnormalised forward DFT, N points
 *   spectrum.c:23-34   fftshift, |X|^2, accumulate, DC-position patch
 *   cbb_main.c:48-59   "zero a row, add K frames"
 *   cbb_main.c:112-128 10*log10(|g * P / K|) -> float dB and/or truncated+clamped u8
 *
 * Geometry of one stream:  output row r accumulates the K frames that start at sample
 *   r * row_hop + j * hop,  j = 0..K-1   (reference: hop = N, K <= 6, row_hop = one source
 *   buffer cadence; per-frame spectra: K = 1, row_hop = hop = N; 50% overlap: hop = N/2).
 * hop and row_hop must be multiples of 8 samples (16-byte TMA alignment).
 */
typedef struct b200_spectrum_plan b200_spectrum_plan;

#define B200_WINDOW_RECT 0   /* the reference */
#define B200_WINDOW_HANN 1   /* periodic Hann, extension */

/* N: a power of two in [16, 65536] (1024, 2048, 4096, 8192 and 65536 have specialised kernels).  gain_db follows cbb_main.c:112 (integer division by 10). */
b200_spectrum_plan* b200_spectrum_plan_create(int N, int hop, int K, int64_t row_hop, int window, int gain_db);
void b200_spectrum_plan_destroy(b200_spectrum_plan* plan);
/* Rows that fit in a stream of n_samples. */
int64_t b200_spectrum_plan_rows(const b200_spectrum_plan* plan, int64_t n_samples);

/*
 * Device-resident execution.  d_iq: interleaved u8 IQ (cmplx_u8 layout, common_sp.h:7-11),
 * stream s starts at d_iq + s * stream_stride_bytes (16-byte aligned).  Outputs are
 * [n_streams][n_rows][N] in display order (index 0 = -fs/2, N/2 = DC position), any of them
 * may be NULL:  d_db float dB, d_power float linear power summed over the K frames (the
 * reference's power_spectrum array), d_db_u8 the payload bytes of cbb_main.c:125-128.
 */
int b200_spectrum_exec(b200_spectrum_plan* plan, const uint8_t* d_iq, int64_t stream_stride_bytes,
                       int n_streams, int64_t n_rows,
                       float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream);

/* Same, for the reference's other two input types (spectrum.c:65-99; no callers in the
 * reference, kept for interface completeness).  cs32: interleaved int32 (re, im), scaled by
 * 1/128 like the u8 path; rf32: real float samples, imaginary part 0, no scaling.
 * Strides are in bytes; frame geometry (hop, row_hop) is in samples of the given type. */
int b200_spectrum_exec_cs32(b200_spectrum_plan* plan, const int32_t* d_iq, int64_t stream_stride_bytes,
                            int n_streams, int64_t n_rows,
                            float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream);
int b200_spectrum_exec_rf32(b200_spectrum_plan* plan, const float* d_x, int64_t stream_stride_bytes,
                            int n_streams, int64_t n_rows,
                            float* d_db, float* d_power, uint8_t* d_db_u8, void* cuda_stream);

/* ---- FM branch: CIC decimation -> discriminator -> two half-band decimators --------------
 *
 * Replaces, fused in one pass over the IQ bytes:
 *   resample.c:6-45     cic_decimate (boxcar sum of R samples minus 128*R, exact int32)
 *   common_sp.h:40-76   atan2_approx
 *   audio_main.c:110-131 first difference (no unwrap) and +-1 hard limiter
 *   resample.c:47-67    halfband_decimate, twice (audio_main.c:133,139)
 * One audio sample per 4*R input samples.
 *
 * State carry: instead of the reference's delay structs (rf_decimator.c:28,
 * audio_main.c:77-79) a stream carries its last b200_fm_history_samples(R) INPUT samples.
 * The caller lays every stream out as [history | batch] and passes the pointer to the batch;
 * a new stream's history is all 128 (b200_fm_history_reset), which reproduces the
 * reference's zero-initialised state exactly, and b200_fm_history_carry copies the batch
 * tail over the history after each batch.  n_samples must be a multiple of 4*R and of 8.
 */
int b200_fm_history_samples(int R);
int b200_fm_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int R, void* cuda_stream);
int b200_fm_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                          int R, void* cuda_stream);
/* The same two calls for a history of any length: history_samples a positive multiple of 8, at most
 * B200_IQ_MAX_HISTORY_SAMPLES (B200_ERR_ARG otherwise); b200_fm_history_reset / _carry are these with 32 R.  Carry needs
 * n_samples >= history_samples. */
#define B200_IQ_MAX_HISTORY_SAMPLES ((1 << 30) - 8)     /* the history's size in bytes stays an int */
int b200_iq_history_reset(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int history_samples,
                          void* cuda_stream);
int b200_iq_history_carry(uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                          int history_samples, void* cuda_stream);
/* d_audio: [n_streams][n_samples / (4R)] floats, row stride audio_stride (floats).
 * d_decimated (nullable): [n_streams][n_samples / R] cmplx_s32, row stride dec_stride (complex). */
int b200_fm_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                 float* d_audio, int64_t audio_stride, int32_t* d_decimated, int64_t dec_stride,
                 void* cuda_stream);

/* ---- FM channels: several stations at frequency offsets inside one dongle's band ----------------
 *
 * The reference demodulates whatever sits at the tuned frequency (resample.c:21-40, audio_main.c:110-139), and
 * its `freq` command retunes the dongle (main.c:139-171), which moves every listener of that dongle.  Here the
 * band stays put and each channel gets the same chain re-centred digitally.  Channel c of stream s has a 32-bit
 * phase increment inc; a signal at baseband +f Hz (RF = dongle frequency + f) is brought to DC by the increment
 * of +f.  With n the int64 index of an input sample from stream start (the history has n < 0):
 *   phi(n) = (uint32)(inc * (uint64) n),   y[n] = ((re - 128) + j (im - 128)) * exp(-j 2 pi phi(n) / 2^32)
 *   b[m]   = sum_{k<R} y[mR + k]           the CIC boxcar of resample.c:21-40 at its own scale, no 1/128
 *   audio  = atan2_approx, first difference, +-1 limiter, two half-bands (audio_main.c:110-139) on b, in f32,
 *            one float per 4R input samples.
 * At inc = 0, b is exactly the integer cic_decimate output and the audio is b200_fm_exec's.  The only state is
 * the input history b200_fm_exec already carries plus the absolute index of the batch's first sample, which the
 * caller passes: an all-128 history mixes to zero, so stream start reproduces the reference's zeroed delay lines.
 * All channels of one call share R.  The filter in front of the demodulator is the reference's boxcar and no
 * sharper: a strong neighbour within fs / R of the channel leaks into it as it would into the reference.
 * b200_fm_channels_exec_fir below replaces the boxcar with a FIR low-pass of up to 1024 taps. */
#define B200_FM_MAX_CHANNELS 32
/* round(offset_hz / sample_rate_hz * 2^32) as a two's-complement uint32; B200_ERR_ARG if |offset| > fs/2, fs <= 0 or NaN.
   Pure host arithmetic: works without a device. */
int b200_fm_channel_tune(double offset_hz, double sample_rate_hz, uint32_t* phase_inc);
/* Layout and history as b200_fm_exec; first_sample >= 0, a multiple of 4R (absolute index of d_iq's first batch sample);
   d_phase_inc: device [n_streams][n_channels]; d_audio row s*n_channels + c (audio_stride floats apart);
   d_baseband (nullable): float (re, im) pairs, row s*n_channels + c, n_samples/R per row, baseband_stride in complex samples.
   n_channels in [1, B200_FM_MAX_CHANNELS], R in [1, 256], n_samples a multiple of 4R and of 8.  Arguments are checked
   before anything is launched: B200_ERR_ARG for counts, R, first_sample, n_samples, NULL pointers, or an audio_stride
   below n_samples/(4R) or a baseband_stride below n_samples/R (the rows would overlap), B200_ERR_ALIGN for
   an IQ pointer or stride that is not 16-byte aligned (or d_audio / d_phase_inc not 4-, d_baseband not 8-byte aligned).
   The audio rows are [n_streams * n_channels][...], so b200_wire_audio_messages turns them into websocket audio
   messages with n_streams * n_channels rows, one per listener; no other wire call is needed. */
int b200_fm_channels_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                          int64_t first_sample, const uint32_t* d_phase_inc, int n_channels,
                          float* d_audio, int64_t audio_stride, float* d_baseband, int64_t baseband_stride,
                          void* cuda_stream);

/* FM channels with a sharper channel filter (opt-in; b200_fm_channels_exec is unchanged).  With y[n] the mixed
 * sample above and h[0..T-1] real taps, the baseband is
 *   b[m] = sum_{k<T} h[k] y[mR + R - T + k]
 * -- the last tap sits on the last sample of the boxcar's window, so T = R with h = 1 IS the boxcar -- decimated by R,
 * and the demodulator after b is the one above.  The filter reaches T - R samples further back than the boxcar, so a
 * stream carries b200_fm_channels_fir_history_samples(R, T) = 32 R + max(T - R, 0), rounded up to a multiple of 8,
 * input samples of history (b200_iq_history_reset / _carry with that length; the layout is [history | batch]).
 * d_taps: T floats on the device, 4-byte aligned, shared by every channel and stream of the call.  T in
 * [1, B200_FM_MAX_CHANNEL_TAPS]; every other argument as b200_fm_channels_exec, and every argument is checked before
 * anything is launched (B200_ERR_ARG for T out of range or NULL d_taps, B200_ERR_ALIGN for a misaligned d_taps).
 * Shared memory: every R in [1, 256] fits with every T up to 1024 (the largest, R = 256 with T = 1024, uses 159 KB for
 * one channel at a time, 212 KB for four).
 * Cost: T taps per decimated sample and channel instead of R (DESIGN.md 4.3b has the measured rates).
 * Taps from b200_fm_channel_filter_design keep the boxcar's DC gain R, so the baseband keeps the scale the
 * demodulator's range assumptions were checked at; any other real taps may be passed.  A signal outside +-fs/2 of
 * the dongle's centre still needs the dongle retuned. */
#define B200_FM_MAX_CHANNEL_TAPS 1024
/* Kaiser-windowed sinc low-pass (host arithmetic, works without a device): n_taps symmetric taps with the -6 dB point
 * at cutoff_hz, Kaiser's beta for atten_db of stopband attenuation, scaled so that the taps sum to R.  B200_ERR_ARG for
 * R outside [1, 256], n_taps outside [1, B200_FM_MAX_CHANNEL_TAPS], cutoff outside (0, fs/2), atten_db negative,
 * fs <= 0, a NaN or infinity, or a NULL h_taps.  Kaiser's estimate of the taps for A dB over a transition of df Hz:
 * n_taps ~= (A - 7.95) / (2.285 * 2 pi df / fs) + 1. */
int b200_fm_channel_filter_design(int R, int n_taps, double cutoff_hz, double atten_db, double sample_rate_hz,
                                  float* h_taps);
/* H(R, T) above; B200_ERR_ARG for R outside [1, 256] or n_taps outside [1, B200_FM_MAX_CHANNEL_TAPS]. */
int b200_fm_channels_fir_history_samples(int R, int n_taps);
int b200_fm_channels_exec_fir(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                              int64_t first_sample, const uint32_t* d_phase_inc, int n_channels,
                              float* d_audio, int64_t audio_stride, float* d_baseband, int64_t baseband_stride,
                              const float* d_taps, int n_taps, void* cuda_stream);

/* FM channels over a ragged table of RUNS: one launch for rows that each have their own channel count, increments and
 * stream position (the push stream's dongles are at different batches and have different listener sets).  Run k
 * demodulates IQ row `stream` (d_iq + stream * stream_stride_bytes, history in front as above) as if it were at
 * absolute sample first_sample, for its n_channels increments; channel c goes to audio row audio_row + c of d_audio
 * (audio_stride floats apart, n_audio_rows rows, each at least n_samples / (4R) floats).  Each run's audio is bit for
 * bit what b200_fm_channels_exec (d_taps == NULL, n_taps == 0) or b200_fm_channels_exec_fir (T = n_taps device taps;
 * the rows then need b200_fm_channels_fir_history_samples(R, T) of history) gives on that row at that position with
 * those increments.  All runs share n_samples and R.  h_runs is host memory, read during the call only.  There is no
 * baseband output.  Checked before anything is launched (B200_ERR_ARG, or B200_ERR_ALIGN for alignment): n_runs in
 * [1, B200_FM_MAX_RUNS]; per run, stream in [0, n_streams), n_channels in [1, B200_FM_MAX_CHANNELS] (a run without
 * channels is left out of the table), first_sample a non-negative multiple of 4R, audio_row >= 0 and
 * audio_row + n_channels <= n_audio_rows; the audio rows of two runs may not overlap; R, n_samples, taps and
 * alignment as for the calls above; n_runs times the tiles of a row below 2^31. */
#define B200_FM_MAX_RUNS 64
typedef struct {
    int32_t stream;                                  /* row of d_iq */
    int32_t n_channels;                              /* [1, B200_FM_MAX_CHANNELS] */
    int64_t first_sample;                            /* >= 0, a multiple of 4R: absolute index of the row's first batch sample */
    int64_t audio_row;                               /* channel c -> audio row audio_row + c */
    uint32_t phase_inc[B200_FM_MAX_CHANNELS];        /* b200_fm_channel_tune */
} b200_fm_channel_run;
int b200_fm_channels_exec_runs(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                               int R, const b200_fm_channel_run* h_runs, int n_runs,
                               float* d_audio, int64_t audio_stride, int64_t n_audio_rows,
                               const float* d_taps, int n_taps, void* cuda_stream);

/* The same demodulator for DECIMATED input -- the signature of the reference's own callback,
 * audio_fm_demodulator(const cmplx_s32*, int) (audio_main.h:12, audio_main.c:74-145), with its three
 * function statics (audio_main.c:77-79) made explicit.  d_state: B200_FM_STATE_FLOATS floats per stream on
 * the device, in/out: [0] previous phase, [1..10] delay_line_1, [11..20] delay_line_2, the rest is the
 * library's; all zero = stream start.  d_decimated: [n_streams][dec_stride] cmplx_s32 (any int32 values:
 * atan2_approx is evaluated in the reference's own order of operations); n_decimated a multiple of 4.
 * Outputs: d_audio n_decimated / 4 floats per stream; optional d_demod (the limiter output of
 * audio_main.c:114-130, n_decimated floats) and d_phase (atan2_approx itself), strides in floats.
 * B200_FM_SKIP_STAGE2 reproduces a block that found the reference's pool full (audio_main.c:137): phase and
 * first half-band advance, the second half-band and its delay line do not, d_audio is not written. */
#define B200_FM_STATE_FLOATS 48
#define B200_FM_SKIP_STAGE2 1
int b200_fm_exec_cs32(const int32_t* d_decimated, int64_t dec_stride, int n_streams, int64_t n_decimated,
                      float* d_state, float* d_audio, int64_t audio_stride, float* d_demod, int64_t demod_stride,
                      float* d_phase, int64_t phase_stride, int flags, void* cuda_stream);
/* Host-buffer form, the body of an rf_decimator_callback: one block of len cmplx_s32 from (borrowed) host
 * memory in, len / 4 audio floats out; h_audio == NULL = B200_FM_SKIP_STAGE2; h_demod nullable.  The state
 * lives in the handle; create = stream start.  libb200audio.so (include/rtlws_audio_compat.h) wraps this in
 * the reference's audio_main.h interface. */
typedef struct b200_fm_demod b200_fm_demod;
b200_fm_demod* b200_fm_demod_create(void);
void b200_fm_demod_destroy(b200_fm_demod* d);
int b200_fm_demod_reset(b200_fm_demod* d);
int b200_fm_demod_block(b200_fm_demod* d, const int32_t* h_signal, int len, float* h_audio, float* h_demod);

/* Diagnostic: atan2_approx (common_sp.h:40-76) as each kernel family evaluates it, on n integer pairs
 * (y, x) -> n floats.  which = 0: the single-quotient form of the FM kernels (|v| < 4096), 1: the folded form
 * of the fused chain kernel, 2: the reference's own order of operations (b200_fm_exec_cs32).  Tests pin all
 * three to the reference's grid. */
int b200_debug_atan2(const int32_t* d_yx, int n, float* d_out, int which, void* cuda_stream);

/* ---- opt-in audio extensions: de-emphasis and 48 kHz output ----------------------------------
 *
 * NOT in the reference (its chain ends at fs / (4R) = 51.2 kS/s without de-emphasis, audio_main.c:133-139,
 * while resources/rtl_ui.js:79-82 wants 48 kHz); off unless asked for, and with flags = 0 nothing changes.
 *   B200_AUDIO_DEEMPH_50US / _75US  y[n] = y[n-1] + alpha (x[n] - y[n-1]), alpha = 1 - exp(-1 / (rate tau))
 *   B200_AUDIO_RESAMPLE_48K         15/16 polyphase FIR (240-tap Blackman-windowed sinc, 16 taps per phase):
 *                                   16 input samples -> 15 output samples; n_audio must be a multiple of 16
 * De-emphasis runs first.  d_state: B200_AUDIO_POST_STATE_FLOATS floats per stream, in/out, zero = stream
 * start.  d_out may not alias d_audio.  The test oracle restates both as plain sequential loops.
 * De-emphasis is computed in parallel: each output is started ceil(ln(1e-7) / ln(1 - alpha)) samples early (at
 * least 96), which grows with audio_rate_hz.  Where that run-in would exceed 1024 samples -- audio_rate_hz above
 * about 850 kHz with 75 us, 1.27 MHz with 50 us -- the call returns B200_ERR_ARG before launching anything. */
#define B200_AUDIO_DEEMPH_50US 1
#define B200_AUDIO_DEEMPH_75US 2
#define B200_AUDIO_RESAMPLE_48K 4
#define B200_AUDIO_POST_STATE_FLOATS 64
int64_t b200_audio_post_out_samples(int64_t n_audio, int flags);
int b200_audio_post(const float* d_audio, int64_t audio_stride, int n_streams, int64_t n_audio, double audio_rate_hz,
                    int flags, float* d_state, float* d_out, int64_t out_stride, void* cuda_stream);
/* The same arithmetic over a table of rows that each name their input, output and state row (the push stream's
 * listeners come and go, and a listener's state belongs to it, not to its position).  Row k reads audio row
 * audio_row of d_audio (audio_stride floats apart, n_audio_rows rows), writes output row out_row of d_out (out_stride
 * floats apart, n_out_rows rows) and advances state row state_row of d_state (B200_AUDIO_POST_STATE_FLOATS floats
 * apart, n_state_rows rows); fresh != 0 reads that state as all zero (stream start) without reading memory.  Row k's
 * output and next state are bit for bit b200_audio_post's on that row with that state (zeroed if fresh), and the
 * state layout is the same, so one state row may be advanced by either call in any order.  h_rows is host memory,
 * read during the call only.  Two launches, like b200_audio_post.  Checked before anything is launched: B200_ERR_ARG
 * for n_rows outside [1, B200_AUDIO_POST_MAX_ROWS], a row index outside its row count, two rows sharing an out_row
 * or a state_row, audio_stride below n_audio or out_stride below b200_audio_post_out_samples(n_audio, flags), NULL
 * pointers, overlapping audio, output and state blocks, and whatever b200_audio_post refuses; B200_ERR_ALIGN for a
 * pointer that is not 4-byte aligned. */
#define B200_AUDIO_POST_MAX_ROWS 1024
typedef struct {
    int32_t audio_row;   /* input row of d_audio */
    int32_t out_row;     /* output row of d_out */
    int32_t state_row;   /* B200_AUDIO_POST_STATE_FLOATS floats at d_state + state_row * that */
    int32_t fresh;       /* nonzero: read the state as all zero (stream start); the next state is written either way */
} b200_audio_post_row;
int b200_audio_post_rows(const float* d_audio, int64_t audio_stride, int64_t n_audio_rows, int64_t n_audio,
                         double audio_rate_hz, int flags, const b200_audio_post_row* h_rows, int n_rows,
                         float* d_state, int64_t n_state_rows, float* d_out, int64_t out_stride, int64_t n_out_rows,
                         void* cuda_stream);
/* the resampler's 240 prototype taps (host), for whoever wants to check them; returns 240 */
int b200_audio_resample_taps(float* h240);

/* ---- the full chain on the same IQ, read once ---------------------------------------------
 *
 * N = 1024 per-frame spectra (K = 1, hop = row_hop = 1024, rectangular: the reference's
 * FFT_POINTS and window) fused with the FM branch at R = 10 (cbb_main.c:80 at 2.048 MS/s).
 * n_samples must be a multiple of 5120 (5 frames = 128 audio samples).  Layout and history
 * as for b200_fm_exec; d_db: [n_streams][n_samples/1024][1024] float dB (display order).
 * d_avg_u8 (nullable): [n_streams][1024] payload bytes of the K_avg-frame average that
 * starts at frame 0 of the batch (the spectrum a UI client would be sent), written
 * directly into the caller's gather/send buffer.
 */
int b200_chain_exec(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples,
                    int gain_db, float* d_db, float* d_audio, int64_t audio_stride,
                    uint8_t* d_avg_u8, int K_avg, void* cuda_stream);
/* The same for any down factor R in [1, 256] (the reference's `bw` command re-derives it as fs / 192000,
 * main.c:152-155, cbb_main.c:80): n_samples must be a multiple of b200_chain_tile_samples(R) = lcm(1024, 4R),
 * history is b200_fm_history_samples(R) samples, d_audio holds n_samples / (4R) floats per stream.  R = 10
 * runs the fused one-pass kernel; other factors run the spectrum and the FM kernel over the same bytes. */
int64_t b200_chain_tile_samples(int R);
int b200_chain_exec_r(const uint8_t* d_iq, int64_t stream_stride_bytes, int n_streams, int64_t n_samples, int R,
                      int gain_db, float* d_db, float* d_audio, int64_t audio_stride,
                      uint8_t* d_avg_u8, int K_avg, void* cuda_stream);

/* ---- host-buffer entry point (what a plugin calls; includes the PCIe copies) --------------
 *
 * Same work as b200_chain_exec for HOST buffers: the library stages the IQ through its own
 * device ring with asynchronous copies on several CUDA streams, runs the kernels and
 * copies the results back.  h_iq: [n_streams][n_samples] cmplx_u8 batch (no history: the
 * session keeps it), h_db / h_audio as above (either may be NULL).  Pinned host memory
 * (b200_host_alloc) makes the copies asynchronous; pageable memory works but serialises.
 */
typedef struct b200_session b200_session;
b200_session* b200_session_create(int n_streams, int64_t max_samples_per_batch);
/* any down factor (b200_session_create is R = 10); batches are multiples of b200_chain_tile_samples(R) */
b200_session* b200_session_create_r(int n_streams, int64_t max_samples_per_batch, int R);
void b200_session_destroy(b200_session* s);
void b200_session_reset(b200_session* s);      /* all streams back to stream start */
int b200_session_chain(b200_session* s, const uint8_t* h_iq, int64_t n_samples, int gain_db,
                       float* h_db, float* h_audio);
/* The same call returning what the reference itself hands its clients instead of per-frame rows: the audio
 * (nullable) and, per stream, the 1024 payload bytes of the K_avg-frame average at the start of the batch
 * (cbb_main.c:40-70 + 106-135; K_avg = 6 is the reference's FFT_AVERAGE).  0.1 B per input sample come back
 * over PCIe instead of 4.1.  h_avg_u8: [n_streams][1024]. */
int b200_session_products(b200_session* s, const uint8_t* h_iq, int64_t n_samples, int gain_db, int K_avg,
                          float* h_audio, uint8_t* h_avg_u8);
/* b200_fm_channels_exec on host buffers: h_phase_inc [n_streams][n_channels] (host), h_audio
 * [n_streams][n_channels][n_samples / (4R)]; batch rules as b200_session_chain.  The session counts the samples
 * every call has consumed (chain, products, channels; b200_session_reset sets it back to 0), so channel calls may
 * be interleaved with the others and each batch is mixed at its absolute position in the stream. */
int b200_session_channels(b200_session* s, const uint8_t* h_iq, int64_t n_samples, const uint32_t* h_phase_inc,
                          int n_channels, float* h_audio);
/* Makes later b200_session_channels calls use the FIR channel filter h_taps (host, n_taps floats; see
 * b200_fm_channels_exec_fir); n_taps = 0 goes back to the boxcar.  Only at stream position 0, i.e. after create or
 * b200_session_reset, like b200_stream_set_payload_sink's "before the first push"; B200_ERR_ARG otherwise, or for n_taps
 * outside [0, B200_FM_MAX_CHANNEL_TAPS], a NULL h_taps with n_taps > 0, or a history
 * b200_fm_channels_fir_history_samples(R, n_taps) longer than the session's max_samples_per_batch.  The session's
 * history grows to that length (the device ring is reallocated and reset), and every later batch of any session call
 * must hold at least that many samples.  Chain and products read only the last 32 R history samples, so their output
 * does not change. */
int b200_session_set_channel_filter(b200_session* s, const float* h_taps, int n_taps);
/* ---- push-style streaming: what a signal_source callback calls ------------------------------
 *
 * signal_source.c:29-35 hands every registered callback a BORROWED buffer of cmplx_u8 and its
 * length (signal_source.h:7).  b200_stream_push is that callback's body: it copies the samples
 * into the stream's pinned host slot and returns; whenever a slot holds `batch_samples`
 * (a multiple of 5120, e.g. the reference's 204800-sample block, rf_decimator.c:65-66) it is
 * submitted asynchronously -- H2D copy, the fused chain kernel, history carry, D2H copies --
 * on one of the library's CUDA streams.  Streams that run in step are submitted together: when every
 * stream of a group of up to 16 consecutive streams has a full slot the group goes out as one copy and
 * one launch; a stream that gets a whole batch ahead of its group goes out alone, and poll / flush submit
 * whatever is waiting.  One producer thread per b200_stream (as the reference has one sensor thread).
 * Finished batches are handed to the sinks from inside push / poll / flush, on the calling thread, in order:
 *   spectrum sink: n_frames rows of 1024 float dB (display order) starting at frame first_frame;
 *   audio sink:    n floats starting at audio sample first_sample: batch_samples / (4R) of them at fs / (4R) (fs/40
 *                  at R = 10), or b200_audio_post_out_samples of that after b200_stream_set_audio_post (below).
 * The pointers passed to a sink are valid until it returns.  Batching is aligned to stream
 * start, so results do not depend on the chunking of the pushes (as with rf_decimator).
 */
typedef struct b200_stream b200_stream;
typedef void (*b200_spectrum_sink)(void* user, int stream, int64_t first_frame, int n_frames, const float* db);
typedef void (*b200_audio_sink)(void* user, int stream, int64_t first_sample, int n, const float* audio);
b200_stream* b200_stream_create(int n_streams, int64_t batch_samples, int gain_db);
/* any down factor (b200_stream_create is R = 10): batch_samples a multiple of b200_chain_tile_samples(R),
 * the audio sink gets batch_samples / (4R) floats per batch at fs / (4R) (unless b200_stream_set_audio_post) */
b200_stream* b200_stream_create_r(int n_streams, int64_t batch_samples, int gain_db, int R);
void b200_stream_destroy(b200_stream* s);
void b200_stream_set_sinks(b200_stream* s, b200_spectrum_sink spectrum_sink, b200_audio_sink audio_sink, void* user);
/* What the reference actually sends its client: the K-frame average at the start of every batch as the 1024 payload
 * bytes of cbb_main.c:121-130 (zero a row, add K frames, 10*log10(|g * P / K|), truncate, clamp), computed on the
 * device (1 KB per batch over PCIe).  With a payload sink and a NULL spectrum sink the per-frame dB rows (4 bytes
 * per sample) stay on the device.  K = 6 is the reference's FFT_AVERAGE (cbb_main.c:18).  Call before the first push. */
typedef void (*b200_payload_sink)(void* user, int stream, int64_t first_frame, int n_frames_averaged, const uint8_t* payload);
int b200_stream_set_payload_sink(b200_stream* s, int K, b200_payload_sink sink);
/* samples: len interleaved (re, im) byte pairs, i.e. a `const cmplx_u8*` */
int b200_stream_push(b200_stream* s, int stream, const uint8_t* samples, int len);
int b200_stream_poll(b200_stream* s);           /* submit what is waiting, deliver what has finished; never blocks */
int b200_stream_flush(b200_stream* s);          /* wait for and deliver every submitted batch */
int64_t b200_stream_pending_samples(const b200_stream* s, int stream);   /* buffered, not yet a whole batch */
/* FM channels on the push stream: listeners at offsets inside each dongle's band (b200_fm_channels_exec).
 * b200_stream_set_channel_sink: up to max_channels ([1, B200_FM_MAX_CHANNELS]) channels per dongle; the first call with
 * a sink allocates the channel audio buffers, a later call with another capacity is refused.  A NULL sink stops channel
 * work: batches submitted without a sink deliver nothing for channels.  The sink gets the `user` of
 * b200_stream_set_sinks and, per batch and channel, n floats at fs / (4R) starting at audio sample first_sample (counted
 * as for the audio sink), after that batch's audio sink call.
 * b200_stream_set_channels replaces dongle `stream`'s listener set (from the stream's producer thread, or serialised
 * with its pushes like any other b200_stream_* call): n_channels increments (b200_fm_channel_tune) and
 * caller-chosen distinct ids, which the sink reports; n_channels = 0 clears the set, and a dongle without channels costs
 * nothing.  B200_ERR_ARG for a bad stream index, n_channels above the capacity, a repeated id or no channel sink.  A batch
 * uses the set that was current when its LAST sample was pushed: a change made while a batch is partly filled
 * (b200_stream_pending_samples) applies to that batch, and a full batch waiting for its group keeps its set.  A channel's
 * audio depends only on the input and its absolute position, so a channel added or retuned at batch b gives exactly
 * what an always-present channel at that offset gives from batch b on.
 * b200_stream_set_channel_filter: the FIR channel filter of b200_fm_channels_exec_fir for every channel of the stream
 * (h_taps: n_taps host floats, n_taps = 0 goes back to the boxcar); only before anything is pushed.  The dongle rows
 * get the history b200_fm_channels_fir_history_samples(R, n_taps); B200_ERR_ARG if that exceeds batch_samples or
 * n_taps is outside [0, B200_FM_MAX_CHANNEL_TAPS].  Spectra, payloads and centre audio do not change. */
typedef void (*b200_channel_audio_sink)(void* user, int stream, int32_t channel_id, int64_t first_sample, int n,
                                        const float* audio);
int b200_stream_set_channel_sink(b200_stream* s, int max_channels, b200_channel_audio_sink sink);
int b200_stream_set_channels(b200_stream* s, int stream, int n_channels, const uint32_t* h_phase_inc,
                             const int32_t* h_channel_ids);
int b200_stream_set_channel_filter(b200_stream* s, const float* h_taps, int n_taps);
/* De-emphasis and 48 kHz output on the push stream (opt-in; flags = 0, the default, leaves every output bit as it
 * was).  flags and audio_rate_hz mean what they mean for b200_audio_post; the rate is fs / (4R), 51200 for the
 * reference.  Only before anything is pushed, like b200_stream_set_channel_filter.  B200_ERR_ARG for whatever
 * b200_audio_post refuses, and for B200_AUDIO_RESAMPLE_48K when batch_samples / (4R) is not a multiple of 16 (every
 * batch at R = 10 is; a batch of 1024 at R = 256 is not).  From then on the audio sink and the channel sink get the
 * post-processed audio: n = b200_audio_post_out_samples(batch_samples / (4R), flags) floats per batch (4800 per
 * 204 800-sample batch with the resampler), first_sample counted at that output rate (batch b starts at b * n).
 * Spectra and payloads do not change.  Each dongle's centre audio carries one state row from stream start.  Each
 * channel carries state by listener id: a listener continues from where it was only if the same id was in the dongle's
 * set in the previous batch and that batch had channel work (a channel sink); any other listener -- a new id, an id
 * back after a gap, every listener of the first batch after batches without a channel sink -- starts from stream-start
 * state.  Retuning an id or reordering the set keeps the state.  Each submitted run adds two launches for the centre
 * audio (b200_audio_post) and, if it has listeners, two for its channels (b200_audio_post_rows). */
int b200_stream_set_audio_post(b200_stream* s, int flags, double audio_rate_hz);

/* ---- websocket wire formats: what the reference's main.c puts on the socket ----------------
 *
 * Replaces the formatting in the LWS_CALLBACK_SERVER_WRITEABLE branch of main.c (a GPU box
 * serving many UI sessions wants what comes back over PCIe to be ready for lws_write):
 *   main.c:80-84   spectrum message  "t s;f %u;b %u;s %d;d" + the payload bytes of
 *                  cbb_get_spectrum_payload (cbb_main.c:106-135), one binary message;
 *   main.c:86-110  audio message  "FF;t a;d" + 8 writes of 2048 bytes of float32 audio
 *                  (first opens a binary message, the rest are continuations, all but the
 *                  last carry NO_FIN): 8 + 16384 bytes once the socket has joined them.
 * Parsed by rtl_ui.js:98-141.  main.c formats the header into a 30-byte stack buffer
 * (main.c:46) and overruns it for 8- and 9-digit frequencies; these functions do not.
 */
#define B200_WIRE_SPECTRUM_HEADER_MAX 48      /* >= the widest "t s;f %u;b %u;s %d;d" (45) */
#define B200_WIRE_AUDIO_FRAGMENTS 8           /* main.c:99-110 */
#define B200_WIRE_AUDIO_FRAGMENT_BYTES 2048   /* main.c:99 */
#define B200_WIRE_AUDIO_MESSAGE_BYTES (8 + B200_WIRE_AUDIO_FRAGMENTS * B200_WIRE_AUDIO_FRAGMENT_BYTES)
/* write flags of a fragment (INTEGRATION.md maps them to LWS_WRITE_BINARY / _CONTINUATION / _NO_FIN) */
#define B200_WIRE_BINARY 1
#define B200_WIRE_CONTINUATION 2
#define B200_WIRE_NO_FIN 0x40
/* audio_get_audio_payload (audio_main.c:40-72) re-sends the first 512 samples of a finished
 * pool buffer in place of the first 512 of the next one.  Off by default; with this flag the
 * emitted sample order is the reference's, byte for byte. */
#define B200_WIRE_REFERENCE_DRAIN 1

/* Header only; returns its length (no terminating NUL is written), B200_ERR_ARG if it does not fit. */
int b200_wire_spectrum_header(char* dst, int dst_len, uint32_t freq_hz, uint32_t sample_rate_hz, int gain_db);
/* Host assembly of one message from host payload bytes; returns the message length. */
int b200_wire_spectrum_message(uint8_t* dst, int dst_len, uint32_t freq_hz, uint32_t sample_rate_hz, int gain_db,
                               const uint8_t* payload, int n_bins);
/* Batched, on the device: message s = header(freq_hz[s], sample_rate_hz[s], gain_db[s]) + the n_bins
 * payload bytes at d_payload + s * payload_stride (what b200_spectrum_exec wrote to d_db_u8 or
 * b200_chain_exec to d_avg_u8), written to d_msgs + s * msg_stride (>= HEADER_MAX + n_bins, bytes
 * past the message up to the next multiple of 4 are zeroed).  freq_hz / sample_rate_hz / gain_db /
 * lens are host arrays; lens[s] (nullable) receives the length.  Strides and pointers: multiples of 4. */
int b200_wire_spectrum_messages(const uint8_t* d_payload, int64_t payload_stride, int n_streams, int n_bins,
                                const uint32_t* freq_hz, const uint32_t* sample_rate_hz, const int32_t* gain_db,
                                uint8_t* d_msgs, int64_t msg_stride, int32_t* lens, void* cuda_stream);
/* Batched audio messages on the device.  Message m of stream s holds wire samples
 * first_wire_sample + 4096 m .. + 4095 of d_audio + s * audio_stride (floats), at
 * d_msgs + s * msg_stride + m * B200_WIRE_AUDIO_MESSAGE_BYTES.  flags = 0: wire sample w is audio
 * sample w.  B200_WIRE_REFERENCE_DRAIN: wire sample w is audio sample
 * b200_wire_reference_drain_index(w, buffer_len) (buffer_len = 5120, audio_main.c:90,100; any multiple of 512 --
 * other pool-buffer lengths make the reference copy partial chunks, which is refused rather than approximated).
 * d_audio must start at the stream's first audio sample in that mode.  first_wire_sample + 4096 n_messages may
 * not exceed audio_stride (the floats a row holds). */
int b200_wire_audio_messages(const float* d_audio, int64_t audio_stride, int n_streams, int64_t first_wire_sample,
                             int n_messages, int flags, int buffer_len, uint8_t* d_msgs, int64_t msg_stride,
                             void* cuda_stream);
/* The lws_write calls of one audio message: fragment `index` (0..7) is `len` bytes at `offset` with `flags`. */
int b200_wire_audio_fragment(int index, int32_t* offset, int32_t* len, int32_t* flags);
int64_t b200_wire_reference_drain_index(int64_t wire_sample, int buffer_len);

/* ---- multi-GPU: stream sharding and the one exchange --------------------------------------
 *
 * All DSP state of the reference is per stream (rf_decimator.c:23,28; audio_main.c:77-79), so streams shard
 * across GPUs with nothing exchanged on the data path: global stream s belongs to rank s mod world, and a
 * rank's streams are its local rows 0, 1, ... in that order (global id = rank + i * world).  The one
 * collective gathers per-stream rows of equal size -- in practice the K-frame averaged payload bytes
 * b200_chain_exec wrote to d_avg_u8, what main.c:80-84 sends a client -- to the rank that serves them.
 * libnccl.so.2 is loaded on first use (NCCL 2.x; a single-GPU host never needs it).
 *
 *   one process per GPU:  rank 0 calls b200_comm_unique_id and hands the 128 bytes to the other ranks by
 *                         whatever the host has (a file, a socket, MPI, torch.distributed); every rank then
 *                         calls b200_comm_create on its own device;
 *   one process, G GPUs:  b200_comm_create_all makes comms[i] for device i; b200_comm_gather_rows_all posts
 *                         the exchange for all of them from one thread.
 *
 * b200_comm_gather_rows: d_send = this rank's local rows [b200_shard_count][row_bytes] (device, contiguous);
 * on the root d_recv receives [n_streams_total][row_bytes] in GLOBAL stream order, other ranks pass NULL.
 * Asynchronous on cuda_stream; row_bytes a multiple of 4.  world == 1 degenerates to a copy. */
#define B200_COMM_ID_BYTES 128
typedef struct b200_comm b200_comm;
int b200_shard_count(int n_streams, int world, int rank);
int b200_shard_stream(int n_streams, int world, int rank, int local_index);
int b200_comm_unique_id(uint8_t* id128);
b200_comm* b200_comm_create(const uint8_t* id128, int world, int rank);
int b200_comm_create_all(int n_devices, b200_comm** comms);
void b200_comm_destroy(b200_comm* c);
int b200_comm_world(const b200_comm* c);
int b200_comm_rank(const b200_comm* c);
int b200_comm_nccl_version(void);       /* e.g. 22703; B200_ERR_CUDA if libnccl cannot be loaded */
int b200_comm_gather_rows(b200_comm* c, const void* d_send, int n_streams_total, int row_bytes, void* d_recv,
                          int root, void* cuda_stream);
int b200_comm_gather_rows_all(b200_comm** comms, int n, const void* const* d_send, int n_streams_total, int row_bytes,
                              void* d_recv, int root, void* const* cuda_streams);

/* One process, G GPUs, HOST buffers: the session above once per device behind one object.  Arrays are in
 * GLOBAL stream order, [n_streams][...]; stream s runs on device s mod n_gpus (its rows are read and
 * written in place with a pitch of n_gpus rows), all devices run concurrently, and h_avg_u8 (nullable;
 * needs K_avg >= 1 at create) receives the K_avg-frame averaged payload bytes of every stream,
 * [n_streams][1024], gathered on device 0 over NCCL first.  R = 10, n_samples a multiple of 5120. */
typedef struct b200_multi b200_multi;
b200_multi* b200_multi_create(int n_gpus, int n_streams, int64_t max_samples_per_batch, int gain_db, int K_avg);
void b200_multi_destroy(b200_multi* m);
int b200_multi_chain(b200_multi* m, const uint8_t* h_iq, int64_t n_samples, float* h_db, float* h_audio,
                     uint8_t* h_avg_u8);

void* b200_host_alloc(uint64_t bytes);          /* pinned host memory */
void b200_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif

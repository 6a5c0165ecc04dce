/*
 * sdr_b200.h -- C ABI of libsdr_b200.so: the B200 (sm_100a) implementation of the
 * sample-stream hot path of agrif/unnamed-rust-sdr.
 *
 * This header is the drop-in boundary.  Every entry point names the reference interface
 * (file:line in the reference tree) it replaces; INTEGRATION.md shows the Rust `extern "C"`
 * block + safe wrappers a maintainer would add.  Conventions (modelled on the reference's one
 * existing FFI, src/resample.rs:33-110 over libsamplerate):
 *   - opaque handles; constructors return NULL and write an error code through `int *err`
 *   - every other call returns an int status, 0 = OK (see sdr_strerror)
 *   - buffers are caller-owned, plain pointers + element counts; nothing is returned allocated
 *   - `*_process` / `*_exec` take HOST pointers (any alignment) and are synchronous
 *   - `*_dev` variants take DEVICE pointers on the handle's device (16-byte aligned) and are
 *     asynchronous on the handle's stream
 *   - a handle is bound to one device + one stream; it may migrate between host threads but
 *     must not be used from two threads at once (Send, not Sync -- resample.rs:25)
 *   - there is NO CPU fallback: without a CUDA device constructors fail with SDR_ERR_NO_DEVICE
 *
 * Sample formats:
 *   SDR_FMT_U8IQ  interleaved u8 I,Q as sent by rtl_tcp; unpacked on the fly exactly as
 *                 RtlTcpSignal::next does: (b as f32 - 128.0) / 128.0   (src/rtltcp.rs:158-164)
 *   SDR_FMT_C64   num::Complex<f32>, interleaved re,im (8 bytes)
 *   SDR_FMT_F32   f32 real samples
 */
#ifndef SDR_B200_H
#define SDR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDR_B200_ABI_VERSION 1

/* ---- status codes ---------------------------------------------------------------------- */
/* 1..22 keep libsamplerate's numbering because src/resample.rs:209-269 hard-codes that map. */
#define SDR_OK 0
#define SDR_ERR_MALLOC_FAILED 1
#define SDR_ERR_BAD_STATE 2
#define SDR_ERR_BAD_DATA 3
#define SDR_ERR_BAD_DATA_PTR 4
#define SDR_ERR_BAD_SRC_RATIO 6
#define SDR_ERR_BAD_CONVERTER 10
#define SDR_ERR_BAD_CHANNEL_COUNT 11
#define SDR_ERR_DATA_OVERLAP 16
#define SDR_ERR_INVALID_ARG 100
#define SDR_ERR_UNSUPPORTED 101
#define SDR_ERR_NO_DEVICE 102
#define SDR_ERR_NULL_HANDLE 103
#define SDR_ERR_OUTPUT_TOO_SMALL 104
#define SDR_ERR_MISALIGNED 105
#define SDR_ERR_CUDA_BASE 1000 /* 1000 + cudaError_t */

const char *sdr_strerror(int code);
int sdr_abi_version(void);
/* number of CUDA devices visible (0 if none / no driver) */
int sdr_device_count(void);
/* name, SM count and memory of device `dev` as a short text line */
int sdr_device_info(int dev, char *buf, size_t cap);

typedef enum { SDR_FMT_U8IQ = 0, SDR_FMT_C64 = 1, SDR_FMT_F32 = 2 } sdr_format_t;

/* ======================================================================================
 * unpack -- RtlTcpSignal::next  (src/rtltcp.rs:158-164).  bit-exact.
 * ====================================================================================== */
int sdr_unpack_u8iq(const uint8_t *iq, size_t n_samples, float *out_c64, int device);
int sdr_unpack_u8iq_dev(const uint8_t *iq, size_t n_samples, float *out_c64, int device, void *stream);

/* ======================================================================================
 * FIR -- filter::Fir<C,A> (src/filter/fir.rs:7-33) driven through signal::Filter
 * (src/signal/adapters/mod.rs:67-100) and, when decimation > 1, signal::Decimate
 * (src/signal/adapters/mod.rs:14-41) fused behind it so that only kept outputs are computed.
 *
 *   y[n] = sum_{k<K} taps[k] * x[n-k],  x[<0] = 0            (fir.rs:23-32)
 *   kept outputs: n = (j+1)*D - 1 over the whole stream      (adapters/mod.rs:30-37)
 * The handle carries the last K-1 inputs and the decimation phase across calls, so feeding a
 * stream in blocks of any size gives the same samples as one call.
 * ====================================================================================== */
/* Default (flags = 0) for u8 IQ input is the integer tcgen05 path: taps are quantised to 24-bit fixed point relative to
 * the largest |tap| (a tap below 2^-24 of the largest contributes nothing; error < 1e-6 of max|y|, see DESIGN.md K5).
 * STRICT_ORDER selects the reference-order CUDA-core kernel instead. */
#define SDR_FIR_STRICT_ORDER 1u /* f32 mul then add, k ascending, no FMA: bit-identical to Fir::apply */
#define SDR_FIR_NO_TENSOR 2u    /* never take a tensor-core path */
#define SDR_FIR_NO_TCGEN05 4u   /* never take the tcgen05/TMEM path (the mma.sync Toeplitz path may still run) */
#define SDR_FIR_SPLIT2 16u      /* c64 input on tcgen05: two bf16 terms per operand (3 products, error < 1e-5 of max|y|) instead of
                                  * three (6 products, the reference's f32 accuracy); ~1.5x less tensor work */
#define SDR_FIR_PLANAR 8u       /* real taps: tcgen05 kernel on de-interleaved I / Q byte planes (same bits; see fir_umma.cu) */

typedef struct {
    const float *taps;   /* n_taps f32, or n_taps (re,im) pairs when taps_complex */
    size_t n_taps;       /* K >= 1 */
    int taps_complex;    /* 0: Fir<f32,A>   1: Fir<Complex<f32>,Complex<f32>> */
    int input_format;    /* sdr_format_t; output is C64 for U8IQ/C64 input, F32 for F32 input */
    size_t decimation;   /* Decimate `wait` D >= 1 (0 is rejected: the reference underflows) */
    size_t n_channels;   /* independent streams sharing the taps (>= 1) */
    unsigned flags;
    int device;
    void *stream;        /* cudaStream_t to run on; NULL = handle creates its own (pass cudaStreamLegacy,
                            (void*)0x1, to run on the legacy default stream) */
} sdr_fir_config_t;

typedef struct sdr_fir sdr_fir_t;
sdr_fir_t *sdr_fir_create(const sdr_fir_config_t *cfg, int *err);
void sdr_fir_destroy(sdr_fir_t *);
int sdr_fir_reset(sdr_fir_t *);                        /* zero history and phase (Fir::new state) */
sdr_fir_t *sdr_fir_clone(const sdr_fir_t *, int *err); /* #[derive(Clone)] on Fir, fir.rs:6 */
/* number of outputs a call with n_in new inputs per channel will produce, given the current phase */
size_t sdr_fir_output_count(const sdr_fir_t *, size_t n_in);
/* in: n_channels rows of n_in elements, row stride in_stride elements (ignored if 1 channel)
 * out: n_channels rows, row stride out_stride elements; out_cap = elements available per row.
 * *n_used = inputs consumed per channel (== n_in on success), *n_out = outputs per channel. */
int sdr_fir_process(sdr_fir_t *, const void *in, size_t n_in, size_t in_stride, void *out,
                    size_t out_cap, size_t out_stride, size_t *n_used, size_t *n_out);
int sdr_fir_process_dev(sdr_fir_t *, const void *in, size_t n_in, size_t in_stride, void *out,
                        size_t out_cap, size_t out_stride, size_t *n_used, size_t *n_out);
/* which kernel family the last process call used: 0 none, 1 CUDA-core direct, 2 CUDA-core
 * strict-order, 3 tensor-core Toeplitz (mma.sync), 4 tensor-core Toeplitz (tcgen05 / TMEM, integer, u8 IQ input),
 * 5 tensor-core Toeplitz (tcgen05 / TMEM, bf16-split operands, c64 input with real taps) */
int sdr_fir_last_path(const sdr_fir_t *);

/* Decimate::new's `wait` = (rate_in / rate_out).round() as usize in f32 (adapters/mod.rs:22) */
size_t sdr_decimate_wait(float rate_in, float rate_out);
/* Take/Skip/Window: (rate * duration).round() as usize (adapters/mod.rs:174,249,279) */
size_t sdr_duration_samples(float rate, float duration);
/* Block: (size * rate).ceil() as usize (adapters/block.rs:117) */
size_t sdr_block_samples(float size, float rate);

/* ======================================================================================
 * FFT -- fft::fft / fft::rfft (src/fft.rs:3-37); the arithmetic replaces rustfft's
 * FFTplanner::plan_fft + process (fft.rs:10-12).
 *   X[k] = sum_n x[n] e^{-2 pi i nk/N}                               (unnormalised forward)
 *   SDR_FFT_SHIFT: out[i] = X[(i - N/2) mod N]                       (fft.rs:15,18-25)
 *   SDR_FFT_NORM : out *= 1.0/(N as f32).sqrt(), multiplied in f32   (fft.rs:16,25)
 *   SDR_FFT_RFFT : input is F32 real, output keeps entries N/2..N-1 of the shifted spectrum
 *                  (rfft's drain(0..len/2), fft.rs:34-36); implies SHIFT
 * A plan is immutable after creation; `batches` consecutive N-point blocks per call.
 * ====================================================================================== */
#define SDR_FFT_SHIFT 1u
#define SDR_FFT_NORM 2u
#define SDR_FFT_RFFT 4u

typedef struct {
    size_t n;          /* transform length: any n >= 1 up to 2^27 (powers of two) or 2^26 (any other length,
                        * Bluestein); SDR_ERR_UNSUPPORTED beyond.  fft::fft takes a whole finite signal */
    int input_format;  /* U8IQ, C64, or F32 (with SDR_FFT_RFFT) */
    unsigned flags;
    int device;
    void *stream;
} sdr_fft_config_t;

typedef struct sdr_fft sdr_fft_t;
sdr_fft_t *sdr_fft_create(const sdr_fft_config_t *cfg, int *err);
void sdr_fft_destroy(sdr_fft_t *);
/* output elements (c64) per transform: n, or n - n/2 with SDR_FFT_RFFT */
size_t sdr_fft_output_len(const sdr_fft_t *);
int sdr_fft_exec(sdr_fft_t *, const void *in, size_t batches, float *out_c64);
/* device pointers: `in` a multiple of the element size (U8IQ 2, C64 8, F32 4 bytes) and `out_c64` of 8 bytes,
 * else SDR_ERR_MISALIGNED before anything runs.  Pointers that meet this but are not 16-byte aligned run kernels
 * without bulk copies. */
int sdr_fft_exec_dev(sdr_fft_t *, const void *in, size_t batches, float *out_c64);
/* the frequency labels of fft.rs:14-24: labels[i] = (i - n/2) as f32 * (rate / n as f32);
 * with rfft != 0 only the kept n - n/2 entries are written.  Host-side, pure. */
int sdr_fft_labels(size_t n, float rate, int rfft, float *labels);

/* ======================================================================================
 * PLL -- filter::Pll / PllDesign (src/filter/pll.rs:4-85) with Biquad / BiquadD / Identity
 * sub-filters (src/filter/biquad.rs:5-154, src/filter/simple.rs:4-19).  One GPU lane per
 * independent stream (the loop itself is sequential).
 * ====================================================================================== */
typedef enum {
    SDR_BQ_IDENTITY = 0, /* filter::Identity */
    SDR_BQ_LOWPASS = 1,  /* BiquadD::LowPass(freq, q)  */
    SDR_BQ_HIGHPASS = 2, /* BiquadD::HighPass(freq, q) */
    SDR_BQ_BANDPASS = 3, /* BiquadD::BandPass(freq, q) */
    SDR_BQ_NOTCH = 4,    /* BiquadD::Notch(freq, q)    */
    SDR_BQ_LR = 5        /* BiquadD::Lr(decayrate)     */
} sdr_biquad_kind_t;

typedef struct { int kind; float p0, p1; } sdr_biquad_design_t;

/* PllDesign::new(reference, gain, loopfilter, outputfilter, lockfilter)  pll.rs:26-36 */
typedef struct {
    float reference, gain;
    sdr_biquad_design_t loopfilter, outputfilter, lockfilter;
} sdr_pll_design_t;

/* BiquadD::design + Biquad::new (biquad.rs:25-38,83-154): coef = b0,b1,b2,na1,na2.  Host, pure. */
int sdr_biquad_design(const sdr_biquad_design_t *d, float rate, float coef[5]);

/* atan2 / sin / cos of the PLL recurrence (pll.rs:72,76).  Default (flags = 0): f32 routines within ~1 ulp of libm's
 * atan2f / sinf / cosf, arranged for the depth of the dependent chain (219 cycles per sample).  SDR_PLL_F64_MATH: the
 * same functions evaluated in f64 and rounded to f32 (equal to libm's result for all but ~1e-4 of the arguments), 455
 * cycles per sample.  Both meet the same parity bars against the CPU oracle (DESIGN.md, K4).  SDR_PLL_FAST_MATH is
 * accepted for source compatibility and has no effect (it selected the f32 routines when f64 was the default). */
#define SDR_PLL_FAST_MATH 1u
#define SDR_PLL_F64_MATH 2u
/* always run the general kernel (per-sample filter-kind tests, fract for any step size) instead of the one specialised
 * for designs without Identity sub-filters and with |reference / rate| + pi |gain| < 1.  Same results bit for bit where
 * both apply (tests/test_gpu_pll_resample.py); for testing. */
#define SDR_PLL_GENERAL_KERNEL 4u

typedef struct {
    const sdr_pll_design_t *designs; /* n_designs entries */
    size_t n_designs;                /* 1 (shared by all streams) or n_streams */
    size_t n_streams;
    float rate;                      /* FilterDesign::design(rate)  pll.rs:48 */
    unsigned flags;
    int device;
    void *stream;
} sdr_pll_config_t;

typedef struct sdr_pll sdr_pll_t;
sdr_pll_t *sdr_pll_create(const sdr_pll_config_t *cfg, int *err);
void sdr_pll_destroy(sdr_pll_t *);
int sdr_pll_reset(sdr_pll_t *);
sdr_pll_t *sdr_pll_clone(const sdr_pll_t *, int *err); /* #[derive(Clone)] pll.rs:12 */
/* in: n_streams rows of n c64 samples (row stride in_stride elements);
 * out: f32 value, locked: 1 iff the reference returns Some(..) (locked > 0.01, pll.rs:80-84) */
int sdr_pll_process(sdr_pll_t *, const float *in_c64, size_t n, size_t in_stride, float *out,
                    uint8_t *locked, size_t out_stride);
int sdr_pll_process_dev(sdr_pll_t *, const float *in_c64, size_t n, size_t in_stride, float *out,
                        uint8_t *locked, size_t out_stride);
/* FM stereo decode around a pilot-tone Pll -- the closure of src/main.rs:62-71:
 *     mono = v * 0.5;  diff = Some(_) = pll.apply(Complex::new(v, 0.0)) ? (v / pll.value.powi(2)).re * 0.5 : 0.0
 * v: n_streams rows of n f32 samples (row stride in_stride samples); out_mono_diff: rows of n
 * (mono, diff) frames (row stride out_stride frames).  Advances the same carried state as process. */
int sdr_pll_stereo_decode(sdr_pll_t *, const float *v, size_t n, size_t in_stride, float *out_mono_diff,
                          size_t out_stride);
int sdr_pll_stereo_decode_dev(sdr_pll_t *, const float *v, size_t n, size_t in_stride, float *out_mono_diff,
                              size_t out_stride);
/* the public fields Pll::nphase / Pll::value (pll.rs:21-22) of one stream; synchronises */
int sdr_pll_get_state(sdr_pll_t *, size_t stream_index, float *nphase, float *value_re, float *value_im);

/* ======================================================================================
 * Biquad as a stream filter -- Filter::apply of filter::Biquad<f32, A> (src/filter/biquad.rs:40-56)
 * driven by signal::Filter (src/signal/adapters/mod.rs:94-96), e.g. the Lr de-emphasis filters of
 * src/main.rs:52,75-80.  A = f32 or Complex<f32> (both parts filtered independently with the
 * same real coefficients).  n_streams independent streams, one GPU lane per real sequence; the
 * operation order of biquad.rs:44-49 is kept (no FMA), so results are bit-identical.
 * ====================================================================================== */
typedef struct {
    const sdr_biquad_design_t *designs; /* n_designs entries */
    size_t n_designs;                   /* 1 (shared by all streams) or n_streams */
    size_t n_streams;
    float rate;                         /* FilterDesign::design(rate), biquad.rs:83 */
    int sample_complex;                 /* 0: Biquad<f32,f32>, 1: Biquad<f32,Complex<f32>> */
    int device;
    void *stream;
} sdr_biquad_config_t;

typedef struct sdr_biquad sdr_biquad_t;
sdr_biquad_t *sdr_biquad_create(const sdr_biquad_config_t *cfg, int *err);
void sdr_biquad_destroy(sdr_biquad_t *);
int sdr_biquad_reset(sdr_biquad_t *);                        /* zero x1, x2, y1, y2 (Biquad::new, biquad.rs:25-38) */
sdr_biquad_t *sdr_biquad_clone(const sdr_biquad_t *, int *err); /* #[derive(Clone)] biquad.rs:4 */
/* in / out: n_streams rows of n samples (f32 or c64), row strides in samples (ignored for one stream) */
int sdr_biquad_process(sdr_biquad_t *, const float *in, size_t n, size_t in_stride, float *out, size_t out_stride);
int sdr_biquad_process_dev(sdr_biquad_t *, const float *in, size_t n, size_t in_stride, float *out, size_t out_stride);

/* ======================================================================================
 * channelizer -- n_channels x ( Fir<f32,Complex<f32>> -> Pll ): config C4.  The FIR output
 * feeds the PLL on chip; only the PLL output leaves.  Same carried state as the two parts.
 * ====================================================================================== */
typedef struct sdr_channelizer sdr_channelizer_t;
sdr_channelizer_t *sdr_channelizer_create(const sdr_fir_config_t *fir, const sdr_pll_config_t *pll, int *err);
void sdr_channelizer_destroy(sdr_channelizer_t *);
int sdr_channelizer_reset(sdr_channelizer_t *);
int sdr_channelizer_process(sdr_channelizer_t *, const void *in, size_t n, size_t in_stride, float *out,
                            uint8_t *locked, size_t out_stride);
int sdr_channelizer_process_dev(sdr_channelizer_t *, const void *in, size_t n, size_t in_stride,
                                float *out, uint8_t *locked, size_t out_stride);

/* ======================================================================================
 * resample -- resample::SampleRate<A> (src/resample.rs:11-110) binds libsamplerate's
 * src_new / src_process / src_reset / src_clone / src_delete / src_set_ratio /
 * src_get_channels / src_strerror (resample.rs:36,61,73,81,105,95,89,196).  The functions
 * below have the same signatures and struct layout, so resample.rs only changes its `use`.
 * Arithmetic: the "sdr-src" specification in DESIGN.md (libsamplerate itself is not in the
 * reference tree: parity unpinned).
 * ====================================================================================== */
enum {
    SDR_SRC_SINC_BEST_QUALITY = 0,
    SDR_SRC_SINC_MEDIUM_QUALITY = 1,
    SDR_SRC_SINC_FASTEST = 2,
    SDR_SRC_ZERO_ORDER_HOLD = 3,
    SDR_SRC_LINEAR = 4
};

typedef struct { /* == libsamplerate SRC_DATA, built at resample.rs:49-58 */
    const float *data_in;
    float *data_out;
    long input_frames, output_frames;
    long input_frames_used, output_frames_gen;
    int end_of_input;
    double src_ratio;
} SDR_SRC_DATA;

typedef struct sdr_src SDR_SRC_STATE;
SDR_SRC_STATE *sdr_src_new(int converter_type, int channels, int *error);
/* same, choosing device/stream (sdr_src_new uses device 0 and its own stream) */
SDR_SRC_STATE *sdr_src_new_on(int converter_type, int channels, int device, void *stream, int *error);
SDR_SRC_STATE *sdr_src_delete(SDR_SRC_STATE *);
int sdr_src_process(SDR_SRC_STATE *, SDR_SRC_DATA *);
/* data_in / data_out are device pointers; counts are still returned synchronously (they are
 * computed on the host), the samples land asynchronously on the handle's stream */
int sdr_src_process_dev(SDR_SRC_STATE *, SDR_SRC_DATA *);
int sdr_src_reset(SDR_SRC_STATE *);
SDR_SRC_STATE *sdr_src_clone(SDR_SRC_STATE *, int *error);
int sdr_src_set_ratio(SDR_SRC_STATE *, double new_ratio);
int sdr_src_get_channels(SDR_SRC_STATE *);
/* frames of input history the handle carries between calls (sinc converters: bounded by the filter
 * wing + what the last call consumed; a call that stops at `output_frames` hands the input it did
 * not need back through input_frames_used, as libsamplerate's src_process does) */
long sdr_src_history_frames(SDR_SRC_STATE *);
/* Sinc converters, long calls (>= 8192 output frames) at an integer step 1/ratio on 2-channel (c64) data run as a
 * polyphase decimating FIR on the tensor cores: within 1e-5 of max|y| of the converter's f64 specification.
 * exact != 0 keeps the f64 kernels for every call (equal to the specification up to the final f32 rounding). */
int sdr_src_set_exact(SDR_SRC_STATE *, int exact);
const char *sdr_src_strerror(int error);
const char *sdr_src_get_name(int converter_type);        /* resample.rs:125 */
const char *sdr_src_get_description(int converter_type); /* resample.rs:133 */
const char *sdr_src_get_version(void);                   /* resample.rs:5 */
/* the windowed-sinc half table of a sinc converter (host pointer, half_len + 2 entries) */
size_t sdr_src_sinc_table(int converter_type, const float **table, int *increment);

/* ======================================================================================
 * stream timing helper for benchmarks: CUDA-event time of everything queued on the handle's
 * stream between begin and end (ms).  Pure measurement, no effect on results.
 * ====================================================================================== */
typedef struct sdr_timer sdr_timer_t;
sdr_timer_t *sdr_timer_create(int device, void *stream, int *err);
void sdr_timer_destroy(sdr_timer_t *);
int sdr_timer_begin(sdr_timer_t *);
int sdr_timer_end(sdr_timer_t *, float *elapsed_ms); /* synchronises the stream */
/* count of kernels this library has launched in this process (all handles) */
uint64_t sdr_kernel_launch_count(void);

/* ======================================================================================
 * FM broadcast stereo receiver -- the signal chain of src/main.rs:32-81 for a batch of
 * stations, every intermediate device-resident:
 *   u8 IQ (rtltcp.rs:158-164) -> Pll demodulator (main.rs:41-49) -> / 75000 -> resample_with(
 *   SincFastest, 144 kHz) (main.rs:50) -> pilot Pll + (mono, diff) decode (main.rs:54-71) ->
 *   resample(48 kHz) (main.rs:73) -> Lr de-emphasis + (mono+diff, mono-diff) (main.rs:52,75-80).
 * Carried state: both PLLs, both converters and the de-emphasis filters of every station, so a
 * stream may be fed in calls of any size.
 * ====================================================================================== */
typedef struct {
    size_t n_stations;
    float rate;     /* input sample rate; main.rs:32 uses 1 800 000 */
    float pilot;    /* pilot tone in Hz; 0 selects main.rs:54's 19 000 */
    unsigned flags; /* SDR_PLL_F64_MATH */
    int device;
    void *stream;
} sdr_fm_config_t;

typedef struct sdr_fm sdr_fm_t;
sdr_fm_t *sdr_fm_create(const sdr_fm_config_t *cfg, int *err);
void sdr_fm_destroy(sdr_fm_t *);
int sdr_fm_reset(sdr_fm_t *);
float sdr_fm_output_rate(const sdr_fm_t *);          /* 48000 */
/* the out_cap sdr_fm_process[_dev] requires for n input samples: a smaller one is rejected with
 * SDR_ERR_OUTPUT_TOO_SMALL before any state changes (the call can be retried with a larger buffer) */
size_t sdr_fm_max_output(const sdr_fm_t *, size_t n);
/* iq: n_stations rows of n u8 IQ samples (2n bytes each, row stride in_stride BYTES);
 * out: n_stations rows of (left, right) f32 frames at 48 kHz, capacity out_cap frames per row,
 * row stride out_stride frames; *n_out = frames written per row (the same for every station).
 * end_of_input != 0 flushes the converters the way signal::Resample does at the end of its
 * upstream (adapters/resample.rs:45-65).  _dev: iq / out are device pointers, rows 16-byte
 * aligned (in_stride % 16 == 0 when n_stations > 1), samples land asynchronously on the stream. */
int sdr_fm_process(sdr_fm_t *, const uint8_t *iq, size_t n, size_t in_stride, float *out, size_t out_cap,
                   size_t out_stride, size_t *n_out, int end_of_input);
int sdr_fm_process_dev(sdr_fm_t *, const uint8_t *iq, size_t n, size_t in_stride, float *out, size_t out_cap,
                       size_t out_stride, size_t *n_out, int end_of_input);

/* ======================================================================================
 * sliding-window spectra -- the spectrum path of examples/live.rs:30-39:
 *     sig.window(duration).decimate(fps).map(|w| fft::fft(from_iter(rate, w...)))
 * Window (src/signal/adapters/mod.rs:271-303) holds the last `window` samples (initially
 * zeros) and yields after every input sample; Decimate (mod.rs:14-41) keeps every hop-th, so
 * kept window j ends at input sample (j + 1) * hop - 1; each kept window goes through
 * fft::fft (src/fft.rs:3-28; flags as sdr_fft_config_t, any length).
 *   window = sdr_duration_samples(rate, duration),  hop = sdr_decimate_wait(rate, fps)
 * Carried state: the last window - 1 samples and the stream position.
 * ====================================================================================== */
typedef struct {
    size_t window;    /* samples per window = transform length */
    size_t hop;       /* Decimate's wait D >= 1 */
    int input_format; /* U8IQ or C64 */
    unsigned flags;   /* SDR_FFT_SHIFT | SDR_FFT_NORM */
    int device;
    void *stream;
} sdr_window_fft_config_t;

typedef struct sdr_window_fft sdr_window_fft_t;
sdr_window_fft_t *sdr_window_fft_create(const sdr_window_fft_config_t *cfg, int *err);
void sdr_window_fft_destroy(sdr_window_fft_t *);
int sdr_window_fft_reset(sdr_window_fft_t *);
size_t sdr_window_fft_size(const sdr_window_fft_t *);
/* windows the next n_in input samples complete */
size_t sdr_window_fft_output_count(const sdr_window_fft_t *, size_t n_in);
/* out_c64: *n_windows consecutive spectra of `window` c64 values each (capacity out_cap windows) */
int sdr_window_fft_process(sdr_window_fft_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                           size_t *n_windows);
int sdr_window_fft_process_dev(sdr_window_fft_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                               size_t *n_windows);

/* ======================================================================================
 * polyphase filter bank -- one wideband stream cut into M channels, each decimated by D.
 * Channel k is filter::Fir<Complex<f32>, Complex<f32>> (src/filter/fir.rs:23-32) with taps
 * g_k[n] = h[n] e^{+2 pi i k n / M} followed by signal::Decimate with wait D (adapters/mod.rs:30-37):
 *   y_k[m] = sum_{n<L} g_k[n] x[(m+1) D - 1 - n],   x[<0] = 0
 * Channel k is centred on k * rate / M; k >= M/2 are the negative frequencies.  Computed as the
 * polyphase form (branch p = taps h[t M + p]) followed by an unnormalised M-point forward DFT
 * (the sdr_fft plan), so accuracy is the FFT's (DESIGN.md).
 *   SDR_PFB_SHIFT          row i of a frame is channel (i - M/2) mod M, at sdr_fft_labels(M, rate, 0)[i]
 *   SDR_PFB_CHANNEL_MAJOR  M rows of frames (what sdr_fir / sdr_pll / sdr_channelizer take as
 *                          n_channels rows) instead of frames of M channels
 *   SDR_PFB_GENERAL_KERNEL always the general front end instead of the register-window one (which runs
 *                          when D divides M and the windows fit in registers); same bits; for testing
 * Carried state: the last L - 1 inputs and the stream position, so blocks of any size give the same
 * bits as one call.  Input pointers need only element alignment (2 bytes u8, 8 bytes c64).
 * ====================================================================================== */
#define SDR_PFB_SHIFT 1u
#define SDR_PFB_CHANNEL_MAJOR 2u
#define SDR_PFB_GENERAL_KERNEL 4u

typedef struct {
    const float *taps;  /* real prototype lowpass h, n_taps f32 */
    size_t n_taps;      /* L >= 1 */
    size_t n_channels;  /* M, 2 <= M <= 65536 (any length the FFT plan accepts) */
    size_t decimation;  /* D >= 1 (0 is rejected, as for sdr_fir) */
    int input_format;   /* U8IQ or C64 (F32 is rejected) */
    unsigned flags;     /* SDR_PFB_* */
    int device;
    void *stream;
} sdr_pfb_config_t;

typedef struct sdr_pfb sdr_pfb_t;
sdr_pfb_t *sdr_pfb_create(const sdr_pfb_config_t *cfg, int *err);
void sdr_pfb_destroy(sdr_pfb_t *);
int sdr_pfb_reset(sdr_pfb_t *);                        /* zero history and stream position */
sdr_pfb_t *sdr_pfb_clone(const sdr_pfb_t *, int *err);
/* frames the next n_in input samples complete */
size_t sdr_pfb_output_count(const sdr_pfb_t *, size_t n_in);
/* frame-major: out = frames of M c64, frame stride out_stride elements (>= M), capacity out_cap frames;
 * channel-major: M rows, row stride out_stride elements (>= frames written), out_cap frames per row.
 * A too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  *n_frames = frames written. */
int sdr_pfb_process(sdr_pfb_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap, size_t out_stride,
                    size_t *n_frames);
int sdr_pfb_process_dev(sdr_pfb_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap, size_t out_stride,
                        size_t *n_frames);

/* ======================================================================================
 * digital down-converter bank -- C channels at arbitrary centre frequencies of one IQ stream, each
 * mixed to 0 Hz by its own 64-bit NCO, low-pass filtered by its own real taps and decimated by D.
 * Channel k restates what the crate builds from a tee'd copy of the stream (Block::clone, adapters/block.rs),
 * a caller-written oscillator through Signal::map, filter::Fir<Complex<f32>, f32> (src/filter/fir.rs:23-32)
 * with taps h_k and signal::Decimate with wait D (adapters/mod.rs:30-37):
 *   z_k[n] = x[n] e^{-2 pi i phi_k(n) / 2^64},   phi_k(n) = (first_sample + n) phase_inc[k]  mod 2^64
 *   y_k[m] = sum_{j<L} h_k[j] z_k[(m+1) D - 1 - j],   x[<0] = 0 (byte 128 for u8, as fir.rs:15)
 * n counts the handle's inputs; first_sample only places the NCO phase (exact 64-bit phase accumulator, so the phase
 * at any stream position is independent of how the stream is cut, across calls and shards).  Channel k is centred on
 * (int64)phase_inc[k] / 2^64 * rate; sdr_ddc_phase_increment(freq, rate) rounds a frequency to an increment:
 * nu = freq / rate, nu -= round(nu), phase_inc = llround(nu 2^64), nu = +-0.5 -> 2^63 (0 for non-finite input).
 * Paths (sdr_ddc_last_path): 2 = tcgen05 integer Toeplitz GEMM for u8 IQ input with D in {1, 2, 4, 8, 16, 32} and
 * L <= 511 while one channel's table fits in shared memory (all but D = 1 with L > ~430); 1 = CUDA-core kernel for
 * everything else (c64 input, other D, longer filters) and with SDR_DDC_GENERAL_KERNEL.  Both meet the FIR bar of
 * 1e-5 of max|y| per channel; they are not bit-equal to each other.
 * Output: C rows (channel-major, the n_channels rows sdr_fir / sdr_pll / sdr_channelizer take), row stride out_stride
 * c64 elements (>= outputs written), out_cap outputs per row; a too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL
 * before any state changes.  Carried state: the last L - 1 inputs and the stream position, so blocks of any size from
 * any element-aligned address give the same bits as one call.
 * ====================================================================================== */
#define SDR_DDC_GENERAL_KERNEL 1u /* always the CUDA-core kernel (for testing; results within the same bars) */

typedef struct {
    const float *taps;         /* n_tap_sets rows of n_taps real f32 */
    size_t n_taps;             /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;         /* 1 (shared) or n_channels */
    const uint64_t *phase_inc; /* n_channels NCO increments (sdr_ddc_phase_increment) */
    size_t n_channels;         /* C, 1 <= C <= 256 (SDR_ERR_INVALID_ARG beyond) */
    size_t decimation;         /* D >= 1 (0 is rejected, as for sdr_fir) */
    uint64_t first_sample;     /* absolute stream index of the first input this handle sees (NCO phase only) */
    int input_format;          /* U8IQ or C64 (F32 is rejected) */
    unsigned flags;            /* SDR_DDC_* */
    int device;
    void *stream;
} sdr_ddc_config_t;

typedef struct sdr_ddc sdr_ddc_t;
uint64_t sdr_ddc_phase_increment(double freq, double rate); /* host, pure */
sdr_ddc_t *sdr_ddc_create(const sdr_ddc_config_t *cfg, int *err);
void sdr_ddc_destroy(sdr_ddc_t *);
int sdr_ddc_reset(sdr_ddc_t *); /* zero history, position back to first_sample */
sdr_ddc_t *sdr_ddc_clone(const sdr_ddc_t *, int *err);
/* outputs per channel that the next n_in input samples complete */
size_t sdr_ddc_output_count(const sdr_ddc_t *, size_t n_in);
int sdr_ddc_process(sdr_ddc_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap, size_t out_stride,
                    size_t *n_out);
int sdr_ddc_process_dev(sdr_ddc_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap, size_t out_stride,
                        size_t *n_out);
int sdr_ddc_last_path(const sdr_ddc_t *); /* path of the last call that produced outputs: 0 none, 1 CUDA-core, 2 tcgen05 */

/* ======================================================================================
 * averaged power spectra -- tapered, overlapped |FFT|^2 of one IQ stream, averaged over K frames.  Restates the
 * crate chain window -> decimate -> map(fft::fft) -> |.|^2 -> mean of K (examples/live.rs:30-39 plus the power
 * and mean a spectrum display computes): Window (adapters/mod.rs:271-303) and Decimate (mod.rs:14-41) give frame
 * j = the N samples ending at input sample (j+1) H - 1, x[<0] = 0 (the deque's initial zeros; frames overlap when
 * H < N and skip samples when H > N), and
 *   X_j[k] = sum_n w[n] frame_j[n] e^{-2 pi i k n / N}        (times 1/sqrt(N) with SDR_PSD_NORM)
 *   P_g[k] = (1/K) sum_{j = gK}^{gK+K-1} |X_j[k]|^2           (f32 rows; K = 1 is a waterfall)
 * Summation order (part of the definition, so outputs are bit-identical however the stream is cut): group g is
 * split into chunks of 32 consecutive frames anchored on its first frame; a chunk sums |X_j[k]|^2 in f32 in
 * ascending j; the chunk partials are summed in f64 in chunk order, scaled by 1/K (and 1/N for NORM) in f64 and
 * rounded to f32 once.
 *   SDR_PSD_SHIFT          bin order of sdr_fft_labels(N, rate, 0)
 *   SDR_PSD_NORM           the 1/sqrt(N) of sdr_fft, i.e. rows scaled by 1/N
 *   SDR_PSD_GENERAL_KERNEL always path 1 (for testing; same bars, not bit-equal to path 2)
 * Paths (sdr_psd_last_path): 2 = one fused kernel (1024-point warp FFT, |X|^2 accumulated in registers) plus a
 * small f64 reduce, for N = 1024 and u8 / c64 input; 1 = gather and taper into L2-sized slabs, sdr_fft plan,
 * accumulate, for every other N (any length sdr_fft_create accepts, Bluestein included).  Both meet the FFT bar
 * carried through |.|^2: |P - P_f64| <= 2e-5 log2(N) max P per row.
 * Carried state: the samples of the pending chunk's frames, the open group's f64 accumulator and the stream
 * position.  The block and the carried tail are read through two pointers (the block is never copied); input
 * pointers need only element alignment (2 bytes u8, 8 bytes c64).
 * ====================================================================================== */
#define SDR_PSD_SHIFT 1u
#define SDR_PSD_NORM 2u
#define SDR_PSD_GENERAL_KERNEL 4u

typedef struct {
    size_t n;             /* N >= 1, any length sdr_fft_create accepts */
    size_t hop;           /* H >= 1 (0 is rejected, as for Decimate) */
    size_t average;       /* K >= 1 */
    const float *window;  /* N real taper values, or NULL = rectangular; copied at create */
    int input_format;     /* U8IQ or C64 (F32 is rejected) */
    unsigned flags;       /* SDR_PSD_* */
    int device;
    void *stream;
} sdr_psd_config_t;

typedef struct sdr_psd sdr_psd_t;
sdr_psd_t *sdr_psd_create(const sdr_psd_config_t *cfg, int *err);
void sdr_psd_destroy(sdr_psd_t *);
int sdr_psd_reset(sdr_psd_t *); /* stream position, carried samples and open group back to the start */
sdr_psd_t *sdr_psd_clone(const sdr_psd_t *, int *err);
/* spectra the next n_in input samples complete */
size_t sdr_psd_output_count(const sdr_psd_t *, size_t n_in);
/* out: spectra of N f32, row stride out_stride floats (>= N), capacity out_cap spectra; a too-small out_cap returns
 * SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  *n_spectra = spectra written. */
int sdr_psd_process(sdr_psd_t *, const void *in, size_t n_in, float *out, size_t out_cap, size_t out_stride,
                    size_t *n_spectra);
/* device pointers, asynchronous on the handle's stream */
int sdr_psd_process_dev(sdr_psd_t *, const void *in, size_t n_in, float *out, size_t out_cap, size_t out_stride,
                        size_t *n_spectra);
int sdr_psd_last_path(const sdr_psd_t *); /* path of the last call that ran frames: 0 none, 1 plan + slab, 2 fused */

/* ======================================================================================
 * fast-convolution channel bank -- sdr_ddc's channels with one decimation per channel, computed by overlap-save, so
 * that the cost barely depends on the filter length and is the same for u8 and c64 input.  Channel k restates a tee'd
 * copy of the stream, a caller-written oscillator (Signal::map), filter::Fir<Complex<f32>, f32> (src/filter/fir.rs:23-32)
 * with taps h_k and signal::Decimate with wait D_k (adapters/mod.rs:30-37); F = first_sample:
 *   z_k[n] = x[n] e^{-2 pi i phi_k(F + n) / 2^64},   phi_k(N) = N phase_inc[k]  mod 2^64
 *   y_k[m] = sum_{j<L} h_k[j] z_k[(m+1) D_k - 1 - j],   x[<0] = 0 (byte 128 for u8, as fir.rs:15)
 * With every D_k = D this is sdr_ddc's function.  Computed in the rotated-taps form by overlap-save on blocks of the
 * ABSOLUTE stream grid: Dl = lcm(D_k), N = the smallest power of two >= 1024 with hop P = floor((N - L + 1) / Dl) Dl
 * >= N / 2 (sdr_fcfb_geometry; SDR_ERR_UNSUPPORTED when N would exceed 2^22).  Block b holds the outputs at absolute
 * indices [b P + eps, (b+1) P + eps), eps = F mod Dl, and is computed from the N inputs that end at its last output:
 * one N-point FFT shared by all channels, a per-channel spectral multiply folded by the power-of-two part of D_k, one
 * small inverse FFT per channel and an exact 64-bit NCO derotation.
 * Release: a block's outputs are written by the call that delivers its last input, so outputs come up to P - 1 samples
 * later than sdr_ddc releases them; sdr_fcfb_output_count gives the per-channel counts.  To drain a finite stream, feed
 * N zeros (the n_fft of sdr_fcfb_geometry) after it and drop the outputs past the stream's end.
 * Bits: an output depends only on its block's N samples and its absolute position, so blockings (1-sample calls, calls
 * that end mid-block), addresses and clones give the bits of one call.  A shard gives the same bits when it is cut on a
 * block boundary of the absolute grid, its halo is at least N - P rounded up to a multiple of Dl, and its first_sample
 * is the halo's absolute index.  A non-finite sample poisons every output, in every channel, of each block whose span
 * holds it, and no other output.
 * Accuracy: per channel |y - y_f64| <= 2e-5 log2(N) max|y_f64| on signals that fill the channel; FFT round-off follows
 * the block's total power, |y_k - y_f64| <~ 1e-7 log2(N) ||h_k||_2 rms(block) (DESIGN.md K9).
 * Output: C rows (channel-major), row stride out_stride c64 elements (>= the largest count), out_cap outputs per row;
 * a too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  *n_out receives C counts.
 * Carried state: fewer than N raw inputs and the stream position; the block and the carried tail are read through two
 * pointers (the block is never copied); input pointers need only element alignment (2 bytes u8, 8 bytes c64).
 * ====================================================================================== */
typedef struct {
    const float *taps;         /* n_tap_sets rows of n_taps real f32 */
    size_t n_taps;             /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;         /* 1 (shared) or n_channels */
    const uint64_t *phase_inc; /* n_channels NCO increments (sdr_ddc_phase_increment) */
    const size_t *decimation;  /* n_channels decimations D_k >= 1 */
    size_t n_channels;         /* C, 1 <= C <= 256 */
    uint64_t first_sample;     /* absolute stream index of the first input: NCO phase and block grid */
    int input_format;          /* U8IQ or C64 (F32 is rejected) */
    int device;
    void *stream;
} sdr_fcfb_config_t;

typedef struct sdr_fcfb sdr_fcfb_t;
/* host, pure: the transform size N and hop P the bank uses for these taps and decimations */
int sdr_fcfb_geometry(size_t n_taps, const size_t *decimation, size_t n_channels, size_t *n_fft, size_t *hop);
sdr_fcfb_t *sdr_fcfb_create(const sdr_fcfb_config_t *cfg, int *err);
void sdr_fcfb_destroy(sdr_fcfb_t *);
int sdr_fcfb_reset(sdr_fcfb_t *); /* carried samples dropped, position back to first_sample */
sdr_fcfb_t *sdr_fcfb_clone(const sdr_fcfb_t *, int *err);
/* counts[k] = channel k's outputs in the blocks that the next n_in input samples complete (C entries) */
int sdr_fcfb_output_count(const sdr_fcfb_t *, size_t n_in, size_t *counts);
int sdr_fcfb_process(sdr_fcfb_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap, size_t out_stride,
                     size_t *n_out);
/* device pointers, asynchronous on the handle's stream */
int sdr_fcfb_process_dev(sdr_fcfb_t *, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                         size_t out_stride, size_t *n_out);

/* ======================================================================================
 * polyphase synthesis filter bank -- M channel streams recombined into one wideband stream at D times
 * the frame rate; the inverse of sdr_pfb.  Channel k (sample m, k < M) is zero-stuffed by D with sample
 * m at index (m+1) D - 1, filtered by filter::Fir<Complex<f32>, Complex<f32>> (src/filter/fir.rs:23-32)
 * with taps f_k[n] = f[n] e^{+2 pi i k n / M}, and all channels are summed:
 *   xh[t] = sum_m sum_k f_k[t - (m+1) D + 1] y_k[m],   0 <= t - (m+1) D + 1 < L
 * Computed in polyphase form: V_m[r] = Y_m[(-r) mod M] with Y_m the unnormalised forward M-point DFT of
 * frame m (the sdr_fft plan), then
 *   xh[t] = sum_{n < L, n = t+1 (mod D)} f[n] V_{(t+1-n)/D - 1}[n mod M]
 * as one fmaf chain per component in ascending n (a tap of 0.0 is still multiplied, so NaNs propagate
 * exactly), frames before the stream being zero.  Accuracy is the FFT's (DESIGN.md).
 * Release: frame m completes outputs [m D, (m+1) D), so n frames give exactly n D outputs; the filter
 * tail comes out when ceil((L-1)/D) zero frames follow.  There is no scale: with an analysis prototype
 * h and a synthesis prototype f of unit DC gain, f must carry a factor D for unit round-trip gain.
 *   SDR_PFS_SHIFT          row i of a frame is channel (i - M/2) mod M, as SDR_PFB_SHIFT writes it
 *   SDR_PFS_CHANNEL_MAJOR  M rows of frames, row stride in_stride (>= frames given), as
 *                          SDR_PFB_CHANNEL_MAJOR writes them; otherwise frames of M, frame stride
 *                          in_stride (>= M).  Both flags only permute on load: every layout gives the same bits
 *   SDR_PFS_GENERAL_KERNEL always the general back end instead of the register-window one (which runs when
 *                          D divides M, M / D <= 8 and ceil(L/D) <= 32); same bits; for testing
 * Carried state: the transforms of the last ceil((L-1)/D) frames, so calls of any number of frames give
 * the same bits as one call.  Pointers need c64 (8-byte) alignment.
 * ====================================================================================== */
#define SDR_PFS_SHIFT 1u
#define SDR_PFS_CHANNEL_MAJOR 2u
#define SDR_PFS_GENERAL_KERNEL 4u

typedef struct {
    const float *taps;     /* real synthesis prototype f, n_taps f32 */
    size_t n_taps;         /* L >= 1 */
    size_t n_channels;     /* M, 2 <= M <= 65536 (any length the FFT plan accepts) */
    size_t interpolation;  /* D >= 1 (0 is rejected) */
    unsigned flags;        /* SDR_PFS_* */
    int device;
    void *stream;
} sdr_pfs_config_t;

typedef struct sdr_pfs sdr_pfs_t;
sdr_pfs_t *sdr_pfs_create(const sdr_pfs_config_t *cfg, int *err);
void sdr_pfs_destroy(sdr_pfs_t *);
int sdr_pfs_reset(sdr_pfs_t *);                        /* zero carried frames */
sdr_pfs_t *sdr_pfs_clone(const sdr_pfs_t *, int *err);
/* outputs that n_frames frames release: n_frames * D */
size_t sdr_pfs_output_count(const sdr_pfs_t *, size_t n_frames);
/* in: n_frames c64 frames, frame-major (frame stride in_stride >= M) or channel-major (M rows, row stride
 * in_stride >= n_frames).  out: n_frames * D c64 samples, capacity out_cap samples.  A too-small out_cap
 * returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  *n_out = samples written. */
int sdr_pfs_process(sdr_pfs_t *, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                    size_t out_cap, size_t *n_out);
int sdr_pfs_process_dev(sdr_pfs_t *, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                        size_t out_cap, size_t *n_out);

/* ======================================================================================
 * digital up-converter bank -- C channel streams, each interpolated by I, mixed up to its own 64-bit-NCO offset and
 * summed into one IQ stream; the transpose of sdr_ddc.  Channel k restates zero-stuffing on sdr_pfs's grid,
 * filter::Fir<f32, Complex<f32>> (src/filter/fir.rs:23-32) with real taps h_k, an oscillator through Signal::map and
 * a sample-by-sample sum; F = first_sample is the absolute stream index of the handle's first OUTPUT:
 *   s_k[(m+1) I - 1] = y_k[m], 0 elsewhere          (m counts the handle's frames; frames before the stream are 0)
 *   u_k[n] = sum_{j<L} h_k[j] s_k[n - j]
 *   x[n]   = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64},   phi_k(N) = N phase_inc[k]  mod 2^64
 * The mixer is the conjugate of sdr_ddc's, so baseband in channel k lands at (int64)phase_inc[k] / 2^64 * rate.
 * Computed with n = q I + c - 1 as u_k[n] = sum_i h_k[c + i I] y_k[q - 1 - i], one fmaf chain per component in
 * ascending i (a tap of 0.0 is still multiplied, so NaNs propagate), then rotated by the exact integer phase and
 * accumulated over ascending k.
 * Release: frame m completes outputs [m I, (m+1) I), so n frames give exactly n I outputs; ceil((L-1)/I) zero frames
 * drain the tail.  There is no scale: for unit round-trip gain after sdr_ddc the synthesis taps carry the factor I.
 * Round trip: after sdr_ddc (first_sample F) and a filter cascade that delays the signal by d samples, give this bank
 * first_sample F - d, or channel k comes back rotated by e^{+2 pi i d phase_inc[k] / 2^64}.
 * Bits: an output depends only on its frames and on F + n, so blockings, clones and shards give the bits of one call.
 * A shard primed with the H = ceil((L-1)/I) frames before it, with first_sample the absolute index of the primed
 * frame's first output, gives one stream's bits after its first H I outputs.
 * Accuracy: |x - x_f64| <= 1e-5 max|x_f64| (DESIGN.md K11).
 * Input: C rows of n_frames c64, row stride in_stride elements (>= n_frames when C > 1): the channel-major rows
 * sdr_ddc and sdr_fcfb write.  Carried state: the last ceil((L-1)/I) frames of every channel and the stream position;
 * the block and the carried frames are read through two pointers (the block is never copied).  Device pointers need
 * c64 (8-byte) alignment.
 * ====================================================================================== */
typedef struct {
    const float *taps;         /* n_tap_sets rows of n_taps real f32 */
    size_t n_taps;             /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;         /* 1 (shared) or n_channels */
    const uint64_t *phase_inc; /* n_channels NCO increments (sdr_ddc_phase_increment) */
    size_t n_channels;         /* C, 1 <= C <= 256 */
    size_t interpolation;      /* I >= 1 (0 is rejected) */
    uint64_t first_sample;     /* absolute stream index of the first OUTPUT (NCO phase only) */
    unsigned flags;            /* 0 */
    int device;
    void *stream;
} sdr_duc_config_t;

typedef struct sdr_duc sdr_duc_t;
sdr_duc_t *sdr_duc_create(const sdr_duc_config_t *cfg, int *err);
void sdr_duc_destroy(sdr_duc_t *);
int sdr_duc_reset(sdr_duc_t *); /* zero carried frames, position back to first_sample */
sdr_duc_t *sdr_duc_clone(const sdr_duc_t *, int *err);
/* outputs that n_frames frames release: n_frames * I */
size_t sdr_duc_output_count(const sdr_duc_t *, size_t n_frames);
/* in: C rows of n_frames c64 samples, row stride in_stride.  out: n_frames * I c64 samples, capacity out_cap samples.
 * A too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  *n_out = samples written. */
int sdr_duc_process(sdr_duc_t *, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                    size_t out_cap, size_t *n_out);
/* device pointers, asynchronous on the handle's stream */
int sdr_duc_process_dev(sdr_duc_t *, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                        size_t out_cap, size_t *n_out);

/* ======================================================================================
 * fast-convolution synthesis bank -- sdr_duc's function with one interpolation per channel, computed by overlap-save,
 * so that the cost barely depends on the filter length; the inverse of sdr_fcfb.  F = first_sample is the absolute
 * stream index of the handle's first OUTPUT:
 *   s_k[(m+1) I_k - 1] = y_k[m], 0 elsewhere          (m counts the handle's frames; frames before the stream are 0)
 *   u_k[n] = sum_{j<L} h_k[j] s_k[n - j]
 *   x[n]   = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64},   phi_k(N) = N phase_inc[k]  mod 2^64
 * With every I_k = I this is sdr_duc's function.  Computed rotate-first: each frame is rotated by its exact integer
 * phase, then x = sum_k g_k * w_k with sdr_fcfb's rotated taps g_k[j] = h_k[j] e^{+2 pi i (j phase_inc[k] mod 2^64)
 * / 2^64}, by overlap-save on sdr_fcfb's geometry (sdr_fcfb_geometry with the interpolations in place of the
 * decimations): Il = lcm(I_k), N, P.  Block b holds the outputs at absolute indices [b P + eps, (b+1) P + eps),
 * eps = F mod Il, and is computed from the frames in the N positions that end at its last output: per channel one
 * small forward FFT of the block's frames, a spectral multiply unfolded by the power-of-two part of I_k and summed over
 * channels, and one N-point inverse FFT shared by all channels.
 * Release: a call advances the handle by n_time output positions (a multiple of Il; row k holds n_time / I_k frames)
 * and writes the outputs of the blocks it completes, up to P - Il positions later than sdr_duc releases them;
 * sdr_fcsb_output_count gives the count.  To drain a finite stream, feed zero frames covering N positions (rounded up
 * to a multiple of Il) and drop the outputs past the stream's end.
 * Bits: an output depends only on its block's frames and its absolute position, so blockings (calls of a single Il,
 * calls that end mid-block), clones and resets give the bits of one call.  A shard gives the same bits when it is cut
 * on a block boundary of the absolute grid, is primed with frames covering at least N - P positions (rounded up to a
 * multiple of Il) and its first_sample is the absolute index of the halo's first output position.  A non-finite frame
 * poisons every output of each block whose span holds it, and no other output.
 * Accuracy: |x - x_f64| <= 2e-5 log2(N) max|x_f64| on signals that fill the channels; FFT round-off follows the total
 * power of the block's frames over all channels, not the level of one channel (DESIGN.md K12).
 * Scale and round trip as sdr_duc: there is no scale (the synthesis taps carry the factor I_k); after sdr_fcfb
 * (first_sample F) and a filter cascade that delays the signal by d samples, give this bank first_sample F - d.
 * sdr_fcfb's per-channel output rows of one call are a valid input of one call at the same stride.
 * Input: C rows, row k = n_time / I_k c64 frames, row stride in_stride c64 (>= the longest row when C > 1).
 * Output: one contiguous c64 stream, out_cap samples; a too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any
 * state changes.  Carried state: the frames of each channel from the next block's span on (fewer than N + Il
 * positions) and the stream position; the caller's rows and the carried frames are read through two pointers (the
 * rows are never copied, except for that tail).  Device pointers need c64 (8-byte) alignment.
 * ====================================================================================== */
typedef struct {
    const float *taps;           /* n_tap_sets rows of n_taps real f32 */
    size_t n_taps;               /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;           /* 1 (shared) or n_channels */
    const uint64_t *phase_inc;   /* n_channels NCO increments (sdr_ddc_phase_increment) */
    const size_t *interpolation; /* n_channels I_k >= 1; N, P = sdr_fcfb_geometry(n_taps, interpolation, C) */
    size_t n_channels;           /* C, 1 <= C <= 256 */
    uint64_t first_sample;       /* absolute stream index of the first OUTPUT: NCO phase and block grid */
    int device;
    void *stream;
} sdr_fcsb_config_t;

typedef struct sdr_fcsb sdr_fcsb_t;
sdr_fcsb_t *sdr_fcsb_create(const sdr_fcsb_config_t *cfg, int *err);
void sdr_fcsb_destroy(sdr_fcsb_t *);
int sdr_fcsb_reset(sdr_fcsb_t *); /* carried frames dropped, position back to first_sample */
sdr_fcsb_t *sdr_fcsb_clone(const sdr_fcsb_t *, int *err);
/* outputs of the blocks that the next n_time output positions complete */
size_t sdr_fcsb_output_count(const sdr_fcsb_t *, size_t n_time);
/* in: C rows, row k = n_time / I_k frames, row stride in_stride c64 (>= the longest row when C > 1).  n_time must be a
 * multiple of lcm(I_k).  *n_out = samples written. */
int sdr_fcsb_process(sdr_fcsb_t *, const float *in_c64, size_t n_time, size_t in_stride, float *out_c64,
                     size_t out_cap, size_t *n_out);
/* device pointers, asynchronous on the handle's stream */
int sdr_fcsb_process_dev(sdr_fcsb_t *, const float *in_c64, size_t n_time, size_t in_stride, float *out_c64,
                         size_t out_cap, size_t *n_out);

/* ======================================================================================
 * rational resampler bank -- C independent c64 channel streams, channel k resampled by its own I_k / D_k with its own
 * real taps h_k: the textbook upfirdn.  Channel k restates sdr_pfs's / sdr_duc's zero-stuffing grid,
 * filter::Fir<f32, Complex<f32>> (src/filter/fir.rs:23-32) and signal::Decimate (adapters/mod.rs:30-37); m counts the
 * handle's frames of the channel and frames before the stream are 0:
 *   s_k[(m+1) I_k - 1] = y_k[m], 0 elsewhere
 *   u_k[n] = sum_{j<L} h_k[j] s_k[n - j]
 *   z_k[r] = u_k[(r+1) D_k - 1]
 * Computed form: with t = (r+1) D_k - 1, q = (t+1) div I_k and c = (t+1) mod I_k,
 *   z_k[r] = sum_{i < I_c} h_k[c + i I_k] y_k[q - 1 - i],   I_c = ceil((L - c) / I_k)
 * as one fmaf chain per component in ascending i: a tap of exactly 0.0 is still multiplied (NaNs propagate exactly),
 * taps with j >= L never are, and an output's bits do not depend on tiling, blocking or launch geometry.
 * Reduction is exact: with g = gcd(I, D) the chain of (g I', g D') with taps h has the same terms in the same order as
 * that of (I', D') with taps h[g j]; the bank reduces every channel at create.
 * Counts: after a channel has received n frames in total it has released floor(n I_k / D_k) outputs (exact integer
 * arithmetic); a call's count is the difference of two such floors and depends only on that channel's frames.
 * Shards: a shard cut at frame s with s I_k = 0 (mod D_k) for every channel, primed with H frames, where H is a multiple
 * of lcm_k(D_k / gcd(I_k, D_k)) and at least max_k ceil(L / I_k), gives one stream's bits after its first H I_k / D_k
 * outputs per channel.  There is no NCO, and the output grid is relative to the handle, as for sdr_fir's decimation.
 * Scale: none.  Unit gain needs taps with DC gain I_k, as for sdr_duc.
 * Accuracy: |z_k - z_k,f64| <= 1e-5 max|z_k,f64| (DESIGN.md K13).
 * Input: C rows, row k of n_in[k] c64 frames, row stride in_stride c64 (>= the longest row when C > 1): sdr_fcfb's
 * mixed-rate rows of one call with its counts and out_stride, or sdr_ddc's / sdr_pfb's equal rows with one count
 * repeated.  Output: C rows of row stride out_stride (>= the largest count when C > 1), out_cap outputs per row; a
 * too-small out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes; *n_out receives C counts.
 * Carried state: the last ceil(L' / I') frames of every channel (L' = ceil(L / g)) and the per-channel frame totals;
 * the caller's rows and the carried frames are read through two pointers (the rows are never copied).  One compute
 * launch per call for all channels, and one small launch that updates the carried frames.  Device pointers need c64
 * (8-byte) alignment.
 * ====================================================================================== */
typedef struct {
    const float *taps;           /* n_tap_sets rows of n_taps real f32 */
    size_t n_taps;               /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;           /* 1 (shared) or n_channels; n_tap_sets * n_taps <= 2^26 */
    const size_t *interpolation; /* n_channels I_k, 1 <= I_k <= 2^16 */
    const size_t *decimation;    /* n_channels D_k, 1 <= D_k <= 2^24 */
    size_t n_channels;           /* C, 1 <= C <= 65536 (sdr_pfb's channel-major rows included) */
    int device;
    void *stream;
} sdr_rrb_config_t;

typedef struct sdr_rrb sdr_rrb_t;
sdr_rrb_t *sdr_rrb_create(const sdr_rrb_config_t *cfg, int *err);
void sdr_rrb_destroy(sdr_rrb_t *);
int sdr_rrb_reset(sdr_rrb_t *); /* carried frames dropped, frame counts back to 0 */
sdr_rrb_t *sdr_rrb_clone(const sdr_rrb_t *, int *err);
/* counts[k] = channel k's outputs from its next n_in[k] frames (C entries each) */
int sdr_rrb_output_count(const sdr_rrb_t *, const size_t *n_in, size_t *counts);
int sdr_rrb_process(sdr_rrb_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                    size_t out_cap, size_t out_stride, size_t *n_out);
/* device pointers, asynchronous on the handle's stream */
int sdr_rrb_process_dev(sdr_rrb_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                        size_t out_cap, size_t out_stride, size_t *n_out);

/* ======================================================================================
 * arbitrary-ratio resampler bank -- C independent c64 channel streams, channel k resampled by its own step sigma_k
 * (input frames per output; any ratio, not only small rationals) on an exact time base, with real taps h_k of length L
 * designed at P times the input rate (P a power of two): GNU Radio's pfb_arb_resampler idea, a polyphase prototype
 * with linear interpolation between adjacent phases.  Positions are exact in units of 2^-64 frames (sdr_arb_time_t);
 * m counts the handle's frames of the channel and frames before the stream are 0:
 *   tau_k(r) = tau_k(0) + r sigma_k                                              (exact integer arithmetic)
 *   H_k(t) = (1 - a) h_k[j] + a h_k[j+1],  j = floor(t P), a = t P - j,  0 <= j < L (h_k[L] = 0); 0 otherwise
 *   z_k[r] = sum_{0 <= m <= floor(tau_k(r))} H_k(tau_k(r) - m) y_k[m]
 * Computed form: n0 = floor(tau), f = its 64-bit fraction, p = log2 P, ip = f >> (64 - p) (0 when P = 1),
 * a = ((f << p) >> 40) 2^-24 (exact in f32: the weight sees the position truncated to 2^-(24+p) frames), the table
 * d_k[j] = f32(h_k[j+1] - h_k[j]) computed in f64 at create, c_i = fmaf(a, d_k[iP + ip], h_k[iP + ip]), and
 *   acc = fmaf(c_i, y_k[n0 - i], acc)   for i = 0, 1, ... while iP + ip < L
 * as one fmaf chain per component: frames before the stream are 0 and still multiplied (NaNs propagate exactly), taps
 * past L never are, and an output's bits depend only on its inputs and its absolute position -- not on tiling,
 * blocking or launch geometry.
 * Counts: output r depends on frames <= floor(tau(r)), so after n frames a channel has released #{r : tau(r) < n} =
 * ceil((n - tau(0)) / sigma) when n > tau(0), else 0 (exact integer arithmetic); a call's count is the difference of two
 * such values and depends only on that channel's frames.
 * Relation to sdr_rrb: with P = I, sigma = D / I, r0 = ceil(I / D) - 1 and tau(0) = ((r0+1) D - I) / I, the outputs are
 * sdr_rrb's outputs r >= r0 bit for bit (a = 0); an output whose tau lies in (n-1, n) is released one frame earlier.
 * Retuning: sdr_arb_set_steps gives every channel a new step from its next unreleased output R on,
 * tau(R + e) = tau_old(R) + e sigma_new; released outputs do not change.  reset restores the creation positions and
 * steps, clone copies the current ones.
 * Shards are anchored on outputs: for any R0_k and a common frame f <= min_k(floor(tau_k(R0_k)) - ceil(L / P) + 1), a
 * handle fed the stream from frame f with first positions tau_k(R0_k) - f and the same steps produces outputs R0_k,
 * R0_k + 1, ... of the whole stream bit for bit.
 * Limits: 2^-16 <= sigma <= 2^24, P <= 2^16, L <= 2^20, n_tap_sets L <= 2^26, C <= 65536; position whole parts, frame
 * totals and per-call counts stay below 2^62, else SDR_ERR_INVALID_ARG.
 * Scale: none.  Unit gain needs sum h = P.
 * Accuracy: |z_k - z_k,f64| <= 1e-5 max|z_k,f64| at exact positions (DESIGN.md K14).
 * Input and output rows are sdr_rrb's: C rows, row k of n_in[k] c64 frames, row stride in_stride (>= the longest row
 * when C > 1); C output rows of out_stride (>= the largest count when C > 1), out_cap outputs per row; a too-small
 * out_cap returns SDR_ERR_OUTPUT_TOO_SMALL before any state changes; *n_out receives C counts.
 * Carried state: the last ceil(L / P) frames of every channel, the frame totals and the time base.  One compute launch
 * per call for all channels and one small launch that updates the carried frames.  Device pointers need c64 (8-byte)
 * alignment.
 * ====================================================================================== */
typedef struct {
    uint64_t whole, frac; /* whole + frac / 2^64 input frames */
} sdr_arb_time_t;

typedef struct {
    const float *taps;           /* n_tap_sets rows of n_taps real f32: the prototype at P times the input rate */
    size_t n_taps;               /* L, 1 <= L <= 2^20 */
    size_t n_tap_sets;           /* 1 (shared) or n_channels; n_tap_sets * n_taps <= 2^26 */
    size_t phases;               /* P, a power of two, 1 <= P <= 2^16 */
    const sdr_arb_time_t *step;  /* n_channels steps, 2^-16 <= sigma <= 2^24 */
    const sdr_arb_time_t *first; /* n_channels first positions (whole part < 2^62), or NULL = all 0 */
    size_t n_channels;           /* C, 1 <= C <= 65536 */
    int device;
    void *stream;
} sdr_arb_config_t;

typedef struct sdr_arb sdr_arb_t;
/* host, pure: rate_in / rate_out rounded to the nearest 2^-64 (ties to even); SDR_ERR_INVALID_ARG for a non-finite or
 * non-positive rate or a result outside [2^-16, 2^24] */
int sdr_arb_step(double rate_in, double rate_out, sdr_arb_time_t *step);
sdr_arb_t *sdr_arb_create(const sdr_arb_config_t *cfg, int *err);
void sdr_arb_destroy(sdr_arb_t *);
int sdr_arb_reset(sdr_arb_t *); /* creation positions and steps, frame counts back to 0 */
sdr_arb_t *sdr_arb_clone(const sdr_arb_t *, int *err);
/* n_channels new steps, from each channel's next unreleased output on */
int sdr_arb_set_steps(sdr_arb_t *, const sdr_arb_time_t *steps);
/* counts[k] = channel k's outputs from its next n_in[k] frames (C entries each) */
int sdr_arb_output_count(const sdr_arb_t *, const size_t *n_in, size_t *counts);
int sdr_arb_process(sdr_arb_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                    size_t out_cap, size_t out_stride, size_t *n_out);
/* device pointers, asynchronous on the handle's stream */
int sdr_arb_process_dev(sdr_arb_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                        size_t out_cap, size_t out_stride, size_t *n_out);

/* ======================================================================================
 * symbol timing recovery bank -- C independent c64 channel streams, each with a Gardner timing loop that steers
 * sdr_arb's interpolator on the same exact time base.  Channel k has real taps h_k of length L designed at P = 2^p
 * times the input rate (typically the matched filter, e.g. a root-raised cosine), a nominal symbol period T_k in input
 * frames (sdr_arb_time_t: sdr_arb_step(rate, symbol_rate) gives it), a first on-time position tau_k(0) and a loop
 * {kp, ki, err_max, max_dev}.  Positions are 64.64 values in units of 2^-64 frames; loop quantities are int64 in
 * units of 2^-40 frames, q(x) = (int64) rint(x 2^40) for an f32 x (exact scaling; create guarantees it fits), and
 * V = floor(max_dev T) in those units, exact from the double's binary value.
 * A(t) is sdr_arb's computed form at absolute position t, bit for bit: the same (h, d) table, the same 2^-24-truncated
 * weight and the same fmaf chain; frames before the stream are 0.  With v_0 = 0 and y_{-1} = 0, for s = 0, 1, 2, ...:
 *   T_s       = T + 2^24 v_s                                     (units of 2^-64; |v_s| <= V)
 *   y_s       = A(tau_s)                                         (the output symbol)
 *   m_s       = A(tau_s - floor(T_s / 2))                        (mid-symbol sample, s >= 1)
 *   g         = fl(fl(fl(y_s.re - y_{s-1}.re) m_s.re) + fl(fl(y_s.im - y_{s-1}.im) m_s.im))
 *   e_s       = 0 for s = 0 or a non-finite g, else min(max(g, -err_max), err_max)
 *   v_{s+1}   = clamp(v_s - q(fl(ki e_s)), -V, V)
 *   tau_{s+1} = tau_s + T + 2^24 v_{s+1} - 2^24 q(fl(kp e_s))
 * e_s is Gardner's detector Re{(y_s - y_{s-1}) conj(m_s)}: e > 0 means the on-time sample is late, so both corrections
 * subtract.  Every f32 operation is rounded on its own (nothing is contracted into an FMA), so a float32 restatement
 * reproduces e, v and tau exactly.  A NaN frame makes the symbols whose chains read it NaN; their errors count as 0,
 * so positions stay finite and deterministic.
 * Validity at create, with D = 2^24 q(fl(kp err_max)): 2 D < T - V, so every step tau_{s+1} - tau_s is at least
 * T_min = T - V - D > 0 and every mid sample m_{s+1} lies after tau_s.  Also rejected (SDR_ERR_INVALID_ARG): max_dev
 * outside [0, 0.25], negative or non-finite kp / ki, err_max <= 0 or non-finite, T outside [1, 2^20] frames,
 * fl(ki err_max) >= 2^22 frames, sdr_arb's limits on P, L, C and tap sets, first whole parts >= 2^62.
 * Release: symbol s is released by the first call after which the channel's frame total n satisfies
 * floor(tau_s) < n (its mid sample lies earlier), so with kp = ki = 0 the counts are sdr_arb's #{r : tau(r) < n}.
 * Counts depend on the data: sdr_tsync_max_output gives the host-computable bound ceil(n_in 2^64 / T_min) per channel
 * (every unreleased tau is >= the previous frame total); a call whose out_cap is below the largest bound returns
 * SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  This is the one bank whose counts come from the device:
 * sdr_tsync_process_dev enqueues its work, copies the C counts back and synchronises the handle's stream.
 * Rows are sdr_arb's: C input rows of n_in[k] frames at in_stride (>= the longest row when C > 1), C output rows of
 * out_stride (>= the largest bound when C > 1); pos (the exact tau_s) and err (e_s) share that stride and may be NULL.
 * Outputs of sdr_ddc, sdr_fcfb and sdr_arb (and sdr_pfb's channel-major rows) feed it unchanged.
 * Carried state per channel: the last ceil(L / P) + ceil((T + V) / 2) + 1 frames, tau of the next unreleased symbol,
 * v, y_{s-1} and the frame total.  reset restores the creation state; clone copies the current one, device part
 * included.  A call is at most 2 launches (compute, carry) and one small copy of the counts back.
 * Not shardable by range: the loop is a recurrence, so the bank shards by channel only.
 * Device pointers need c64 (8-byte) alignment for rows and positions, 4 bytes for err.
 * ====================================================================================== */
typedef struct {
    float kp, ki;   /* proportional and integral gains, frames per unit of e (sdr_tsync_loop_design) */
    float err_max;  /* the detector output is clamped to [-err_max, err_max] */
    double max_dev; /* |v| <= max_dev T, 0 <= max_dev <= 0.25 */
} sdr_tsync_loop_t;

typedef struct {
    const float *taps;             /* as sdr_arb_config_t: n_tap_sets rows of n_taps real f32 at P times the rate */
    size_t n_taps, n_tap_sets, phases;
    const sdr_arb_time_t *period;  /* n_channels nominal periods T_k, 1 <= T_k <= 2^20 frames */
    const sdr_arb_time_t *first;   /* n_channels first positions (whole part < 2^62), or NULL = all 0 */
    const sdr_tsync_loop_t *loops; /* n_loops loop parameter sets */
    size_t n_loops;                /* 1 (shared) or n_channels */
    size_t n_channels;             /* C, 1 <= C <= 65536 */
    int device;
    void *stream;
} sdr_tsync_config_t;

typedef struct sdr_tsync sdr_tsync_t;
/* host, pure: gains of the standard second-order (PI, type-2) loop for a noise bandwidth bn_t (normalised to the
 * symbol rate), damping zeta, detector slope ted_gain (mean e per symbol period of timing error) and a period of
 * period_frames input frames:
 *   theta = bn_t / (zeta + 1 / (4 zeta)),  delta = 1 + 2 zeta theta + theta^2,
 *   kp = 4 zeta theta / (delta ted_gain) period_frames,  ki = 4 theta^2 / (delta ted_gain) period_frames
 * in frames per unit of e (this bank's units); SDR_ERR_INVALID_ARG unless every argument is positive and finite */
int sdr_tsync_loop_design(double bn_t, double zeta, double ted_gain, double period_frames, float *kp, float *ki);
sdr_tsync_t *sdr_tsync_create(const sdr_tsync_config_t *cfg, int *err);
void sdr_tsync_destroy(sdr_tsync_t *);
int sdr_tsync_reset(sdr_tsync_t *); /* creation positions, v = 0, y_{-1} = 0, frame totals back to 0 */
sdr_tsync_t *sdr_tsync_clone(const sdr_tsync_t *, int *err);
/* caps[k] = ceil(n_in[k] 2^64 / T_min_k): the most symbols channel k can release from its next n_in[k] frames */
int sdr_tsync_max_output(const sdr_tsync_t *, const size_t *n_in, size_t *caps);
int sdr_tsync_process(sdr_tsync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *sym_c64,
                      sdr_arb_time_t *pos, float *err, size_t out_cap, size_t out_stride, size_t *n_out);
/* device pointers; returns after the counts are copied back (synchronises the handle's stream) */
int sdr_tsync_process_dev(sdr_tsync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *sym_c64,
                          sdr_arb_time_t *pos, float *err, size_t out_cap, size_t out_stride, size_t *n_out);
/* the next unreleased position and the period offset v (2^-40 frames) of one channel; synchronises */
int sdr_tsync_get_state(sdr_tsync_t *, size_t channel, sdr_arb_time_t *next, int64_t *v);

/* ======================================================================================
 * carrier recovery bank -- C independent c64 symbol streams (one sample per symbol, e.g. sdr_tsync's output rows with
 * its counts as n_in), each with a decision-directed Costas loop that removes the carrier frequency and phase left
 * after down-conversion.  State per channel: the phase phi, a uint64 in units of 2^-64 turn (the NCO convention of
 * sdr_ddc), and the frequency nu, an int64 in units of 2^-40 turn per symbol with |nu| <= V = floor(max_freq 2^40)
 * (exact).  q(x) = (int64) rint(x 2^40) for an f32 x.  From phi_0 and nu_0 (config, default 0), for s = 0, 1, 2, ...:
 *   r_s       = nco_rot_fast(phi_s) ~ e^{-2 pi i phi_s / 2^64}
 *   z_s       = (fl(fl(x.re r.re) - fl(x.im r.im)), fl(fl(x.re r.im) + fl(x.im r.re)))     (the output symbol)
 *   e_s       = 0 for a non-finite g = D_M(z_s), else min(max(g, -err_max), err_max)
 *   nu_{s+1}  = clamp(nu_s + q(fl(ki e_s)), -V, V)
 *   phi_{s+1} = phi_s + 2^24 (nu_{s+1} + q(fl(kp e_s)))                                    (mod 2^64)
 * nco_rot_fast(phi): f = fl((float)(int64) phi 2^-64), (s, c) = an f32 sincos of fl(f 6.2831855f) (quadrant from f),
 * r = (c, -s); within a few 1e-7 of the exact rotation.
 * Detectors, with a = sgn(z.re) z.im and b = sgn(z.im) z.re (exact; sgn(x) = +1 for x >= 0, -0 included, else -1) and
 * K = f32(sqrt 2 - 1) -- GNU Radio's order-2/4/8 Costas detectors, order 2 decision-directed:
 *   M = 2  (+-1):                 D = a                                                     slope K_d = A
 *   M = 4  ((+-1 +- i)/sqrt 2):   D = fl(a - b)                                             K_d = sqrt(2) A
 *   M = 8  (e^{i pi (2k+1)/8}):   D = |z.re| >= |z.im| ? fl(a - fl(K b)) : fl(fl(K a) - b)   K_d = A / cos(pi/8)
 * (K_d: mean D per radian of phase error at amplitude A).  e > 0 means z leads its decision, so both corrections add.
 * Every f32 operation is rounded on its own (nothing is contracted into an FMA): a float32 restatement gives e_s from
 * the reported z_s bit for bit, and integer arithmetic every phi_s and nu_s from the reported e_s.  A non-finite x_s
 * gives a non-finite z_s and e_s = 0: nu stays and phi advances by 2^24 nu, so the state stays finite.
 * Loop design: sdr_tsync_loop_design(bn_t, zeta, K_d, 1 / (2 pi)) gives kp and ki in turns per unit of e (the same
 * type-2 loop; 1 / (2 pi) turns per radian takes the place of the period).
 * Validity at create (SDR_ERR_INVALID_ARG): order not 2, 4 or 8; kp or ki negative or non-finite; err_max <= 0 or
 * non-finite; fl(kp err_max) or fl(ki err_max) >= 1 / (2 M) turn (one correction stays within half a decision sector);
 * max_freq outside [0, 1 / (2 M)]; |nu_0| > V; C outside [1, 65536]; n_loops not 1 or C.
 * One symbol out per symbol in: the counts are n_in, so sdr_csync_process_dev copies nothing back and does not
 * synchronise.  Rows: C input rows of n_in[k] symbols at in_stride, C output rows z at out_stride (both >= the longest
 * row when C > 1); phase (phi_s) and err (e_s) rows share out_stride and may be NULL.  out may equal in with the same
 * stride (in place).  reset restores the creation phases and frequencies; clone copies the current ones.  A call is one
 * launch and one small upload of the counts.  The loop is a recurrence, so the bank shards by channel only.
 * Device pointers need 8-byte alignment for rows and phases, 4 bytes for err.
 * ====================================================================================== */
typedef struct {
    unsigned order;  /* M: 2, 4 or 8 (the constellations above) */
    float kp, ki;    /* turns per unit of e: sdr_tsync_loop_design(bn_t, zeta, K_d, 1 / (2 pi)) */
    float err_max;   /* e is clamped to [-err_max, err_max] */
    double max_freq; /* |nu| <= V = floor(max_freq 2^40), 0 <= max_freq <= 1 / (2 M) turns per symbol */
} sdr_csync_loop_t;

typedef struct {
    const sdr_csync_loop_t *loops; /* n_loops loop parameter sets */
    size_t n_loops;                /* 1 (shared) or n_channels */
    const uint64_t *phase;         /* n_channels phi_0 in 2^-64 turns, or NULL = 0 */
    const int64_t *freq;           /* n_channels nu_0 in 2^-40 turns per symbol, or NULL = 0 */
    size_t n_channels;             /* C, 1 <= C <= 65536 */
    int device;
    void *stream;
} sdr_csync_config_t;

typedef struct sdr_csync sdr_csync_t;
sdr_csync_t *sdr_csync_create(const sdr_csync_config_t *cfg, int *err);
void sdr_csync_destroy(sdr_csync_t *);
int sdr_csync_reset(sdr_csync_t *); /* the creation phases and frequencies */
sdr_csync_t *sdr_csync_clone(const sdr_csync_t *, int *err);
int sdr_csync_process(sdr_csync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                      uint64_t *phase, float *err, size_t out_stride);
/* device pointers, asynchronous on the handle's stream */
int sdr_csync_process_dev(sdr_csync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                          uint64_t *phase, float *err, size_t out_stride);
/* phi and nu of one channel's next symbol; synchronises */
int sdr_csync_get_state(sdr_csync_t *, size_t channel, uint64_t *phase, int64_t *freq);

/* ======================================================================================
 * adaptive equalizer bank -- C independent c64 symbol streams (one sample per symbol, e.g. sdr_tsync's output rows with
 * its counts as n_in), each through an N-tap FIR whose complex weights adapt by blind CMA and then decision-directed
 * LMS, to remove the intersymbol interference of multipath and filter mismatch.  One tap count N for the handle,
 * 1 <= N <= 64.  Channel k carries the weights w[0..N), a delay line x_{s-j} (zeros before the stream), a symbol total
 * s and an adaptation set {M, mu, a, err_max, S}: M in {2, 4, 8} (sdr_csync's constellations +-1, (+-1 +- i)/sqrt 2 and
 * e^{i pi (2k+1)/8}, scaled to radius a), the step mu >= 0, the radius a > 0 with R = fl(a a), err_max > 0, and S:
 * symbols s < S adapt by CMA and s >= S by DD (S = UINT64_MAX: CMA only; S = 0: DD only).  For each symbol s:
 *   P_j = w[j] x_{s-j} = (fl(fl(w.re x.re) - fl(w.im x.im)), fl(fl(w.re x.im) + fl(w.im x.re)))
 *   W   = 2^ceil(log2 min(N, 32)) lanes; p_l = P_l for l < min(N, W), 0 for N <= l < W;
 *         N > 32: p_l = fl(P_l + P_{l+32}) where l + 32 < N, else P_l
 *   y_s = pairwise tree over p_0..p_{W-1}: for o = W/2, ..., 1: p_l <- fl(p_l + p_{l+o});  y_s = p_0
 *   CMA: eps = fl(fl(fl(y.re y.re) + fl(y.im y.im)) - R),  g = (fl(eps y.re), fl(eps y.im))
 *   DD:  d = D_M(y) at radius a, g = (fl(y.re - d.re), fl(y.im - d.im)), with sgn(-0) = +1:
 *        M = 2: (+-a, 0);  M = 4: (+-c, +-c), c = f32(a / sqrt 2);
 *        M = 8: |y.re| >= |y.im| ? (+-p, +-q) : (+-q, +-p), p = f32(a cos pi/8), q = f32(a sin pi/8)
 *        (c, p and q computed in double at create and rounded once)
 *   y or g not finite: e_s = 0 and the taps do not change (no update is computed: a NaN in the delay line cannot
 *   reach w); else e_s = each component of g clamped to [-err_max, err_max],  u = (fl(mu e.re), fl(mu e.im)),
 *   w[j] <- (fl(w.re - fl(fl(u.re x.re) + fl(u.im x.im))), fl(w.im - fl(fl(u.im x.re) - fl(u.re x.im))))
 *   (w <- w - mu e conj(x), x = x_{s-j}: the gradient of E(|y|^2 - R)^2 and of E|y - d|^2)
 * Every f32 operation is rounded on its own (nothing is contracted into an FMA) and the summation order is part of the
 * definition, so a numpy float32 restatement reproduces every y_s, every e_s and the final taps bit for bit.
 * Initial taps: n_tap_sets rows of N c64 (1 shared, or C), or n_tap_sets = 0 for the centre spike
 * w[floor((N-1)/2)] = 1, which delays the output by that many symbols; the weights must be finite.
 * Validity at create (SDR_ERR_INVALID_ARG): N outside [1, 64]; C outside [1, 65536]; n_adapt not 1 or C; n_tap_sets
 * not 0, 1 or C; NULL taps with n_tap_sets > 0, or non-finite taps; M not 2, 4 or 8; mu negative or non-finite; a <= 0,
 * non-finite, or with R = fl(a a) not finite; err_max <= 0 or non-finite.
 * One symbol out per symbol in: the counts are n_in, so sdr_eq_process_dev copies nothing back and does not
 * synchronise.  Rows: C input rows of n_in[k] symbols at in_stride, C output rows y and C error rows e (c64, may be
 * NULL) at out_stride (both strides >= the longest row when C > 1).  out may equal in with the same stride (in place).
 * reset restores the creation taps, zeroes the delay lines and sets s = 0; clone copies the current state.  A call is
 * one launch and one small upload of the counts: the taps, the last N - 1 symbols and s live on the device between
 * calls.  The equalizer is a recurrence, so the bank shards by channel only.  Device rows need 8-byte alignment.
 * ====================================================================================== */
typedef struct {
    unsigned order;        /* M: 2, 4 or 8 (the DD decisions above) */
    float mu;              /* step, >= 0 */
    float radius;          /* a > 0: the CMA modulus R = fl(a a) and the DD constellation's radius */
    float err_max;         /* each component of e is clamped to [-err_max, err_max] */
    uint64_t cma_symbols;  /* S: symbols s < S adapt by CMA, s >= S by DD */
} sdr_eq_adapt_t;

typedef struct {
    size_t n_taps;                /* N, 1 <= N <= 64 */
    const float *taps;            /* n_tap_sets rows of N c64, or NULL with n_tap_sets = 0 */
    size_t n_tap_sets;            /* 0 (centre spike), 1 (shared) or n_channels */
    const sdr_eq_adapt_t *adapt;  /* n_adapt adaptation sets */
    size_t n_adapt;               /* 1 (shared) or n_channels */
    size_t n_channels;            /* C, 1 <= C <= 65536 */
    int device;
    void *stream;
} sdr_eq_config_t;

typedef struct sdr_eq sdr_eq_t;
sdr_eq_t *sdr_eq_create(const sdr_eq_config_t *cfg, int *err);
void sdr_eq_destroy(sdr_eq_t *);
int sdr_eq_reset(sdr_eq_t *); /* the creation taps, zero delay lines, s = 0 */
sdr_eq_t *sdr_eq_clone(const sdr_eq_t *, int *err);
int sdr_eq_process(sdr_eq_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                   float *err_c64, size_t out_stride);
/* device pointers, asynchronous on the handle's stream */
int sdr_eq_process_dev(sdr_eq_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                       float *err_c64, size_t out_stride);
/* the N c64 taps of one channel for its next symbol; synchronises */
int sdr_eq_get_taps(sdr_eq_t *, size_t channel, float *taps_c64);

/* ======================================================================================
 * Viterbi decoder bank -- C independent soft-decision streams of one convolutional code, e.g. sdr_csync's output rows
 * (Gray QPSK at rate 1/2: one c64 symbol is one step, I -> c_0, Q -> c_1, in_stride counted in steps).
 * Code: constraint length K, 3 <= K <= 9, S = 2^(K-1) states; rate 1/n, 2 <= n <= 4; generators g_0 .. g_{n-1}, each
 * in [1, 2^K), in the usual octal convention where the MSB taps the current input (802.11: K = 7, (0133, 0171)).
 * Encoder the decoder inverts: the state s_{t-1} holds the K - 1 previous inputs, u_{t-1} at bit K - 2;
 *   r_t = (u_t << (K-1)) | s_{t-1},  c_{t,j} = popcount(r_t & g_j) mod 2,  s_t = r_t >> 1.
 * Soft input: step t reads n f32 values x[t n + j]; a positive value favours bit 0 (BPSK 0 -> +1).  With the scale
 * sigma_k of channel k: a non-finite x gives q = 0 (an erasure), else q = rint(clamp(fl(x sigma_k), -127, 127)),
 * rounding half to even; a product that overflows saturates.  Erasures are how callers depuncture: they insert zeros.
 * Branch cost: sum_j (c_j ? 127 + q_j : 127 - q_j), an integer in [0, 254 n].
 * Add-compare-select: the new state s' has predecessors p_b = ((s' << 1) & (S-1)) | b; m'(s') = min_b m(p_b) + cost;
 * the decision d = 1 only when the b = 1 sum is strictly smaller (ties take b = 0).
 * Start metrics: zero start m(0) = 0 and every other state I = (K-1) 254 n + 1 (after K - 1 steps every survivor
 * descends from state 0); uniform start: every state 0, for a stream picked up mid-way.
 * Release: L is the decision depth, a multiple of 32, 32 <= L <= 512.  At every per-channel step total T = 32 j with
 * T >= L + 32: the best state after step T - 1 (least metric, ties to the lowest index), a traceback through steps
 * T - 1 .. T - L - 32 (step i's bit is s >> (K-2), the previous state ((s << 1) & (S-1)) | d_i(s)), and the bits of
 * steps [T - L - 32, T - L) are released.  After T steps since create, reset or finish E(T) = max(0, 32 floor(T/32) - L)
 * bits are out, so a call's count per channel is E(T + n_in) - E(T): the host knows it without asking the device
 * (sdr_vit_output_count), and sdr_vit_process_dev does not synchronise.
 * Finish: for the channels in `which` (C bytes, nonzero = listed; NULL: all) the T - E(T) <= L + 31 remaining bits by
 * one traceback from state 0 (terminated != 0) or from the best state; the channel then returns to its creation state.
 * Metrics are exact integers (never renormalised); the spread max m - min m never exceeds (2K - 3) 254 n + 1, so the
 * device holds them in 32 bits and compares modulo 2^32 with the same decisions.
 * Validity at create (SDR_ERR_INVALID_ARG): K, n, L or C out of range; a generator 0 or >= 2^K; a scale <= 0 or
 * non-finite; n_scales not 1 and not C.
 * Rows: C input rows of n_in[k] steps (n f32 each) at in_stride steps (>= the longest row when C > 1); C output rows
 * of one byte per decoded bit (0 or 1) at out_stride bytes (>= the largest count when C > 1); n_out receives C counts.
 * Device rows need 4-byte alignment (out_stride a multiple of 4 when C > 1).  reset returns every channel to its
 * creation state; clone copies the current state.  A call is one launch and one small upload of the counts: the
 * metrics, the undecoded decisions and T live on the device.  The decoder is a recurrence, so the bank shards by
 * channel only.
 * ====================================================================================== */
typedef struct {
    unsigned constraint;  /* K, 3..9 */
    const uint32_t *gens; /* n generators, octal convention above */
    size_t n_gens;        /* n, 2..4 */
    size_t depth;         /* L: multiple of 32, 32..512 */
    const float *scale;   /* n_scales soft-value scales sigma_k > 0, finite */
    size_t n_scales;      /* 1 (shared) or n_channels */
    int zero_start;       /* 1: the encoder starts in state 0; 0: uniform start */
    size_t n_channels;    /* C, 1..65536 */
    int device;
    void *stream;
} sdr_vit_config_t;

typedef struct sdr_vit sdr_vit_t;
sdr_vit_t *sdr_vit_create(const sdr_vit_config_t *cfg, int *err);
void sdr_vit_destroy(sdr_vit_t *);
int sdr_vit_reset(sdr_vit_t *); /* every channel to its creation state, T = 0 */
sdr_vit_t *sdr_vit_clone(const sdr_vit_t *, int *err);
/* host only, no device work: n_out[k] = E(T_k + n_in[k]) - E(T_k) */
int sdr_vit_output_count(const sdr_vit_t *, const size_t *n_in, size_t *n_out);
int sdr_vit_process(sdr_vit_t *, const float *in, const size_t *n_in, size_t in_stride, uint8_t *out,
                    size_t out_stride, size_t *n_out);
/* device pointers, asynchronous on the handle's stream; n_out is filled on the host */
int sdr_vit_process_dev(sdr_vit_t *, const float *in, const size_t *n_in, size_t in_stride, uint8_t *out,
                        size_t out_stride, size_t *n_out);
int sdr_vit_finish(sdr_vit_t *, const uint8_t *which, int terminated, uint8_t *out, size_t out_stride, size_t *n_out);
/* device out, asynchronous; n_out is filled on the host */
int sdr_vit_finish_dev(sdr_vit_t *, const uint8_t *which, int terminated, uint8_t *out, size_t out_stride,
                       size_t *n_out);

/* ======================================================================================
 * frame synchronizer bank -- C independent c64 symbol streams (e.g. sdr_csync's output rows), each carrying frames of
 * F symbols that start with a known sync word.  The bank finds the word by correlation, tracks frames with a
 * search -> verify -> lock -> flywheel state machine, reads the constellation's phase ambiguity (sdr_csync locks up to
 * a rotation by 2 pi / M, CMA leaves any phase) from the phase of each frame's correlation, and emits each frame's
 * payload derotated: the input sdr_vit needs, from the library alone.
 * Sync word: one length Lp per handle, 8 <= Lp <= 1024; n_words rows of Lp c64 (1 shared, or C), finite, with
 * E_p > 0 and finite.  Parameters {F, M, th_search, th_check, V, max_miss, W}, 1 set or C: F the frame period in
 * symbols (word included), Lp + 2 W < F <= 2^24; M in {2, 4, 8} (sdr_csync's constellations); th_search, th_check in
 * (0, 1]; V <= 8 verifications before lock; 1 <= max_miss <= 255; W <= 32 the check window half-width.
 * Symbols z_t are numbered from 0 since create or reset; position s reads z_s .. z_{s+Lp-1}.  Every f32 operation is
 * rounded on its own (nothing is contracted):
 *   P_j  = conj(p_j) z_{s+j} = (fl(fl(p.re z.re) + fl(p.im z.im)), fl(fl(p.re z.im) - fl(p.im z.re)))
 *   c_s  = P_0, then c_s <- fl(c_s + P_j) for j = 1 .. Lp-1, componentwise and in that order
 *   E_s  = the same sequential sum of fl(fl(z.re z.re) + fl(z.im z.im)); E_p the same over the word, once
 *   rho_s = fl(a / b) if b > 0, else 0, with a = fl(fl(c.re c.re) + fl(c.im c.im)), b = fl(E_s E_p)
 * A test passes when rho >= theta; a NaN rho fails every test.  The best position of the window around e is the
 * s in [e - W, e + W] with the largest rho_s (NaN lowest), ties to the smallest |s - e|, then to the earlier s.
 * Rotation r(c) in [0, M), sgn(-0) = +1: M = 2: c.re >= 0 ? 0 : 1;  M = 4: q = |c.re| >= |c.im| ? (c.re >= 0 ? 0 : 2)
 * : (c.im >= 0 ? 1 : 3);  M = 8: q as for M = 4, c' = c (-i)^q (exact), t = fl(K c'.re) with K = f32(sqrt 2 - 1),
 * o = c'.im > t ? 1 : (c'.im < -t ? -1 : 0), r = (2 q + o) mod 8.
 * Derotation D_r(x) = x e^{-2 pi i r / M}: sign changes and swaps for M = 2 and 4; for M = 8 and odd r first
 * x <- (fl(fl(x.re + x.im) h), fl(fl(x.im - x.re) h)) with h = f32(1 / sqrt 2), then x (-i)^floor(r / 2), exact.
 * State machine, per channel, decisions in increasing position order, each made once the symbols it needs are in:
 *   SEARCH from sigma: the first s >= sigma with rho_s >= th_search: HIT.  V = 0: LOCK at once, emit the frame at s,
 *           R = r(c_s), e = s + F.  Else VERIFY with e = s + F, v = 0.
 *   VERIFY: s* = the best position around e.  Pass (rho >= th_check): VERIFY_PASS, v += 1; at v = V: LOCK, emit the
 *           frame at s*, R = r(c_s*); either way e = s* + F.  Fail: VERIFY_FAIL, SEARCH from sigma = e + W + 1.
 *   LOCK:   s* = the best position around e.  Pass: LOCK_PASS, R = r(c_s*), m = 0, emit the frame at s*, e = s* + F.
 *           Fail: m += 1; m < max_miss: LOCK_MISS, emit the frame at e with R unchanged (flywheel), e += F;
 *           else LOCK_LOST, SEARCH from sigma = e + W + 1.
 * Emitting the frame at s appends D_R(z_t), t = s + Lp .. s + F - 1, to the channel's payload stream as those symbols
 * arrive: every emitted frame carries F - Lp symbols, and a frame's payload is complete before the next decision.
 * The search never rewinds: positions passed over while verifying are not searched again (the word repeats, so this
 * costs at most one more frame of acquisition).
 * Records (sdr_fsync_record_t), one per decision: pos = s* for HIT and passes, e for fails, misses and losses;
 * out_index = the payload index of the emitted frame's first symbol, or UINT64_MAX when no frame is emitted; corr and
 * rho of the best (or hit) position in every case; rot = the R a frame is emitted with, else r(corr); kind.
 * Bounds (sdr_fsync_max_output, host only): for n_in = n > 0 symbols after T consumed, with G = F - W + 1 and
 * m = 1 if Lp >= W else 2,  payload <= m (n + min(T, Lp + 2 W - 1)),  records <= min(n, 2 floor((n - 1) / G) + 2).
 * Proof: each symbol completes at most one decision; after a fail or a loss the next decision is a HIT, after which
 * the next one completes at least F + W symbols later; after any other decision the next one completes at least
 * F - W symbols later, so any two consecutive gaps sum to at least G.  Emitted frames start at least F - W apart, so
 * a symbol lies in at most m payloads; a call emits its own symbols and, at decisions, carried ones.
 * A call whose out_cap (or rec_cap, when recs is not NULL) is below the largest bound returns
 * SDR_ERR_OUTPUT_TOO_SMALL before any state changes.  Counts depend on the data: like sdr_tsync_process_dev,
 * sdr_fsync_process_dev enqueues its work, copies the C counts back and synchronises the handle's stream.
 * Rows: C input rows of n_in[k] symbols at in_stride (>= the longest row when C > 1); C payload rows at out_stride
 * (>= the largest payload bound when C > 1); recs may be NULL, else C rows of rec_stride records (>= the largest
 * record bound when C > 1); n_rec may be NULL.  Symbol totals stay below 2^62 (else SDR_ERR_INVALID_ARG).
 * Carried per channel: fewer than Lp + 2 W symbols, the state, the totals.  reset returns every channel to SEARCH
 * from 0 with nothing consumed; clone copies the current state, device part included.  A call is one launch, one
 * small upload of the counts and one copy of the C output counts back.  The state machine is a recurrence, so the
 * bank shards by channel only.  Device pointers need 8-byte alignment.
 * ====================================================================================== */
#define SDR_FSYNC_SEARCH 0
#define SDR_FSYNC_VERIFY 1
#define SDR_FSYNC_LOCK 2

#define SDR_FSYNC_HIT 1
#define SDR_FSYNC_VERIFY_PASS 2
#define SDR_FSYNC_VERIFY_FAIL 3
#define SDR_FSYNC_LOCK_PASS 4
#define SDR_FSYNC_LOCK_MISS 5
#define SDR_FSYNC_LOCK_LOST 6

typedef struct {
    uint32_t period;        /* F: frame period in symbols, word included; Lp + 2 W < F <= 2^24 */
    uint32_t order;         /* M: 2, 4 or 8 */
    float thresh_search;    /* th_search in (0, 1] */
    float thresh_check;     /* th_check in (0, 1] */
    uint32_t verify;        /* V <= 8 */
    uint32_t max_miss;      /* 1..255 */
    uint32_t window;        /* W <= 32 */
} sdr_fsync_params_t;

typedef struct {
    size_t word_len;                  /* Lp, 8..1024 */
    const float *words;               /* n_words rows of Lp c64 */
    size_t n_words;                   /* 1 (shared) or n_channels */
    const sdr_fsync_params_t *params; /* n_params parameter sets */
    size_t n_params;                  /* 1 (shared) or n_channels */
    size_t n_channels;                /* C, 1..65536 */
    int device;
    void *stream;
} sdr_fsync_config_t;

typedef struct {
    uint64_t pos;       /* s* for HIT and passes; e for fails, misses and losses */
    uint64_t out_index; /* payload index of the emitted frame's first symbol, or UINT64_MAX */
    float corr[2];      /* c of the best (or hit) position */
    float rho;          /* its rho */
    uint16_t rot;       /* R of the emitted frame, else r(corr) */
    uint16_t kind;      /* SDR_FSYNC_HIT .. SDR_FSYNC_LOCK_LOST */
} sdr_fsync_record_t;

typedef struct {
    uint32_t state;     /* SDR_FSYNC_SEARCH, _VERIFY or _LOCK */
    uint32_t count;     /* v (VERIFY) or m (LOCK) */
    uint64_t pos;       /* sigma (SEARCH) or e */
    uint32_t rot;       /* R */
    uint32_t pad;
    uint64_t consumed;  /* symbols since create or reset */
    uint64_t payload;   /* payload symbols emitted (counting the current frame whole) */
} sdr_fsync_state_t;

typedef struct sdr_fsync sdr_fsync_t;
sdr_fsync_t *sdr_fsync_create(const sdr_fsync_config_t *cfg, int *err);
void sdr_fsync_destroy(sdr_fsync_t *);
int sdr_fsync_reset(sdr_fsync_t *); /* every channel to SEARCH from 0, nothing consumed */
sdr_fsync_t *sdr_fsync_clone(const sdr_fsync_t *, int *err);
/* host only: pay_caps[k], rec_caps[k] = the bounds above for the next n_in[k] symbols of channel k */
int sdr_fsync_max_output(const sdr_fsync_t *, const size_t *n_in, size_t *pay_caps, size_t *rec_caps);
int sdr_fsync_process(sdr_fsync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                      size_t out_cap, size_t out_stride, size_t *n_out, sdr_fsync_record_t *recs, size_t rec_cap,
                      size_t rec_stride, size_t *n_rec);
/* device pointers; returns after the counts are copied back (synchronises the handle's stream) */
int sdr_fsync_process_dev(sdr_fsync_t *, const float *in_c64, const size_t *n_in, size_t in_stride, float *out_c64,
                          size_t out_cap, size_t out_stride, size_t *n_out, sdr_fsync_record_t *recs, size_t rec_cap,
                          size_t rec_stride, size_t *n_rec);
/* one channel's state; synchronises */
int sdr_fsync_get_state(sdr_fsync_t *, size_t channel, sdr_fsync_state_t *state);

#ifdef __cplusplus
}
#endif
#endif /* SDR_B200_H */

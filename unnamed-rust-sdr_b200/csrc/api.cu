// api.cu -- the extern "C" layer of libsdr_b200.so (declared in include/sdr_b200.h).
// Host-side state machines only: stream history, decimation phase, resampler positions, plans.
// All arithmetic on samples happens in the kernels (fir.cu, fft.cu, pll.cu, resample.cu).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"

namespace sdr {
std::atomic<uint64_t> g_launches{0};
}

using namespace sdr;

namespace {

inline size_t elem_bytes(int fmt) { return fmt == SDR_FMT_U8IQ ? 2 : (fmt == SDR_FMT_C64 ? 8 : 4); }
inline size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

// Rust `f32 as usize` (saturating; NaN and negatives -> 0)
inline size_t f32_as_usize(float v) {
    if (!(v > 0.0f)) return 0;
    if (v >= 18446744073709551616.0f) return SIZE_MAX;
    return (size_t)v;
}

int copy2d(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width, size_t height, cudaMemcpyKind kind,
           cudaStream_t st) {
    if (width == 0 || height == 0) return SDR_OK;
    if (height == 1 || (dpitch == width && spitch == width))
        return cuda_status(cudaMemcpyAsync(dst, src, width * height, kind, st));
    return cuda_status(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, kind, st));
}

// Double-buffered host<->device pipeline for the host-pointer entry points: chunk c is uploaded on `up`,
// computed on the handle's stream and downloaded on `down`, so H2D(c+1), kernel(c) and D2H(c-1) overlap
// (PCIe is full duplex).  Events order buffer reuse; nothing here touches sample values.
struct HostPipe {
    cudaStream_t up = nullptr, down = nullptr;
    cudaEvent_t e_up[2] = {nullptr, nullptr}, e_k[2] = {nullptr, nullptr}, e_down[2] = {nullptr, nullptr};
    bool ready = false;
    HostPipe() = default;
    HostPipe(const HostPipe &) = delete;
    HostPipe &operator=(const HostPipe &) = delete;
    ~HostPipe() {
        if (up) cudaStreamDestroy(up);
        if (down) cudaStreamDestroy(down);
        for (int i = 0; i < 2; ++i) {
            if (e_up[i]) cudaEventDestroy(e_up[i]);
            if (e_k[i]) cudaEventDestroy(e_k[i]);
            if (e_down[i]) cudaEventDestroy(e_down[i]);
        }
    }
    int init() {
        if (ready) return SDR_OK;
        SDR_CUDA_TRY(cudaStreamCreateWithFlags(&up, cudaStreamNonBlocking));
        SDR_CUDA_TRY(cudaStreamCreateWithFlags(&down, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            SDR_CUDA_TRY(cudaEventCreateWithFlags(&e_up[i], cudaEventDisableTiming));
            SDR_CUDA_TRY(cudaEventCreateWithFlags(&e_k[i], cudaEventDisableTiming));
            SDR_CUDA_TRY(cudaEventCreateWithFlags(&e_down[i], cudaEventDisableTiming));
        }
        ready = true;
        return SDR_OK;
    }
    // before uploading into buffer b: the kernel that last read it must be done
    int begin_upload(int b) { return cuda_status(cudaStreamWaitEvent(up, e_k[b], 0)); }
    int end_upload(int b) { return cuda_status(cudaEventRecord(e_up[b], up)); }
    // before the kernel on `main` touches buffer b: its upload is done and the download that last read out[b] is done
    int begin_compute(int b, cudaStream_t main) {
        SDR_CUDA_TRY(cudaStreamWaitEvent(main, e_up[b], 0));
        return cuda_status(cudaStreamWaitEvent(main, e_down[b], 0));
    }
    int end_compute(int b, cudaStream_t main) {
        SDR_CUDA_TRY(cudaEventRecord(e_k[b], main));
        return cuda_status(cudaStreamWaitEvent(down, e_k[b], 0));
    }
    int end_download(int b) { return cuda_status(cudaEventRecord(e_down[b], down)); }
    int drain(cudaStream_t main) {
        SDR_CUDA_TRY(cudaStreamSynchronize(down));
        SDR_CUDA_TRY(cudaStreamSynchronize(up));
        return cuda_status(cudaStreamSynchronize(main));
    }
};

}  // namespace

// ============================================================================================
// misc
// ============================================================================================
extern "C" const char *sdr_strerror(int code) {
    switch (code) {
        case SDR_OK: return "No error.";
        case SDR_ERR_MALLOC_FAILED: return "Malloc failed.";
        case SDR_ERR_BAD_STATE: return "SRC_STATE pointer is NULL.";
        case SDR_ERR_BAD_DATA: return "SRC_DATA pointer is NULL.";
        case SDR_ERR_BAD_DATA_PTR: return "SRC_DATA->data_out or SRC_DATA->data_in is NULL.";
        case SDR_ERR_BAD_SRC_RATIO: return "SRC ratio outside [1/256, 256] range.";
        case SDR_ERR_BAD_CONVERTER: return "Bad converter number.";
        case SDR_ERR_BAD_CHANNEL_COUNT: return "Channel count must be >= 1.";
        case SDR_ERR_DATA_OVERLAP: return "Input and output data arrays overlap.";
        case SDR_ERR_INVALID_ARG: return "Invalid argument.";
        case SDR_ERR_UNSUPPORTED: return "Unsupported size or combination.";
        case SDR_ERR_NO_DEVICE: return "No CUDA device available (libsdr_b200 has no CPU fallback).";
        case SDR_ERR_NULL_HANDLE: return "Handle is NULL.";
        case SDR_ERR_OUTPUT_TOO_SMALL: return "Output buffer too small.";
        case SDR_ERR_MISALIGNED: return "Device pointer must be 16-byte aligned.";
        default:
            if (code >= SDR_ERR_CUDA_BASE) return cudaGetErrorString((cudaError_t)(code - SDR_ERR_CUDA_BASE));
            return "Unknown error.";
    }
}
extern "C" int sdr_abi_version(void) { return SDR_B200_ABI_VERSION; }
extern "C" int sdr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
extern "C" int sdr_device_info(int dev, char *buf, size_t cap) {
    int rc = check_device(dev);
    if (rc) return rc;
    cudaDeviceProp p;
    SDR_CUDA_TRY(cudaGetDeviceProperties(&p, dev));
    snprintf(buf, cap, "%s sm_%d%d %d SMs %.1f GiB", p.name, p.major, p.minor, p.multiProcessorCount,
             (double)p.totalGlobalMem / (1024.0 * 1024.0 * 1024.0));
    return SDR_OK;
}
extern "C" uint64_t sdr_kernel_launch_count(void) { return g_launches.load(); }

// adapters/mod.rs:22 : (signal.rate() / rate).round() as usize
extern "C" size_t sdr_decimate_wait(float rate_in, float rate_out) { return f32_as_usize(roundf(rate_in / rate_out)); }
// adapters/mod.rs:174,249,279 : (signal.rate() * duration).round() as usize
extern "C" size_t sdr_duration_samples(float rate, float duration) { return f32_as_usize(roundf(rate * duration)); }
// adapters/block.rs:117 : (size * signal.rate()).ceil() as usize
extern "C" size_t sdr_block_samples(float size, float rate) { return f32_as_usize(ceilf(size * rate)); }

// ============================================================================================
// unpack
// ============================================================================================
extern "C" int sdr_unpack_u8iq_dev(const uint8_t *iq, size_t n, float *out, int device, void *stream) {
    int rc = check_device(device);
    if (rc) return rc;
    DeviceGuard g(device);
    if (!g.ok) return g.status();
    return unpack_launch(iq, n, out, (cudaStream_t)stream);
}
extern "C" int sdr_unpack_u8iq(const uint8_t *iq, size_t n, float *out, int device) {
    int rc = check_device(device);
    if (rc) return rc;
    if (n == 0) return SDR_OK;
    if (!iq || !out) return SDR_ERR_BAD_DATA_PTR;
    DeviceGuard g(device);
    if (!g.ok) return g.status();
    DevBuf din, dout;
    rc = din.reserve(2 * n);
    if (!rc) rc = dout.reserve(8 * n);
    if (!rc) rc = cuda_status(cudaMemcpy(din.p, iq, 2 * n, cudaMemcpyHostToDevice));
    if (!rc) rc = unpack_launch((const uint8_t *)din.p, n, (float *)dout.p, 0);
    if (!rc) rc = cuda_status(cudaMemcpy(out, dout.p, 8 * n, cudaMemcpyDeviceToHost));
    return rc;
}

// ============================================================================================
// FIR
// ============================================================================================
struct FirHost {
    int dev = 0;
    int fmt = 0, taps_complex = 0;
    unsigned flags = 0;
    size_t K = 0, Kp = 0, HL = 0, D = 1, n_ch = 1;
    size_t hist_stride = 0;
    std::vector<float> taps;  // padded host copy
    size_t phase = 0;  // inputs already discarded in the current decimation group
    int last_path = 0;
};

struct sdr_fir : FirHost {
    StreamRef stream;
    DevBuf d_taps;
    DevBuf d_tc_tables;  // tensor-core Toeplitz tap fragments (u8 input, non-strict)
    float tc_scale = 1.0f;
    DevBuf d_uc_tables;  // tcgen05 Toeplitz bf16 tap-term tables (c64 input, real taps, non-strict, D == 1)
    int uc_ns = 0;
    DevBuf d_um_tables;  // tcgen05 Toeplitz digit tables (u8 input, non-strict, D == 1)
    int um_R = 0, um_PC = 0, um_planar = 0, um_magic[2][3] = {{0, 0, 0}, {0, 0, 0}};
    float um_sc[3] = {0.0f, 0.0f, 0.0f};
    DevBuf d_hist[2];
    int cur = 0;
    DevBuf d_in, d_out, d_in2, d_out2;
    HostPipe pipe;

    int alloc(void *user_stream, const sdr_fir *);
    int copy_device(const sdr_fir &src) {
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, n_ch * hist_stride * elem_bytes(fmt),
                                      cudaMemcpyDeviceToDevice));
    }
};

int sdr_fir::alloc(void *user_stream, const sdr_fir *) {
    int rc = stream.init(user_stream);
    if (rc) return rc;
    if ((rc = d_taps.upload(taps.data(), Kp * (taps_complex ? 2 : 1) * sizeof(float), stream.s))) return rc;
    const size_t hbytes = n_ch * hist_stride * elem_bytes(fmt);
    for (int i = 0; i < 2; ++i)
        if ((rc = d_hist[i].alloc(hbytes))) return rc;
    rc = fir_fill_hist(d_hist[0].p, fmt, (long long)(n_ch * hist_stride), stream.s);
    if (rc) return rc;
    if (fmt == SDR_FMT_U8IQ && !(flags & (SDR_FIR_STRICT_ORDER | SDR_FIR_NO_TENSOR)) && K <= 4096 && D <= 64) {
        std::vector<uint2> tab;
        tc_scale = fir_tc_build_tables(taps.data(), (int)K, taps_complex != 0, (int)D, tab);
        if ((rc = d_tc_tables.upload(tab.data(), tab.size() * sizeof(uint2), stream.s))) return rc;
        SDR_CUDA_TRY(cudaStreamSynchronize(stream.s));
    }
    int R = 0, PC = 0, planar = 0;
    if (fmt == SDR_FMT_U8IQ && !(flags & (SDR_FIR_STRICT_ORDER | SDR_FIR_NO_TENSOR | SDR_FIR_NO_TCGEN05)) && D <= (1u << 20) &&
        fir_umma_geometry((int)K, (int)D, taps_complex != 0, (flags & SDR_FIR_PLANAR) != 0, &R, &PC, &planar)) {
        std::vector<uint8_t> tab;
        if (fir_umma_build_tables(taps.data(), (int)K, taps_complex != 0, R, PC, planar, (int)D, tab, um_magic, um_sc)) {
            um_R = R;
            um_PC = PC;
            um_planar = planar;
            if ((rc = d_um_tables.upload(tab.data(), tab.size(), stream.s))) return rc;
            SDR_CUDA_TRY(cudaStreamSynchronize(stream.s));
        }
    }
    if (fmt == SDR_FMT_C64 && !(flags & (SDR_FIR_STRICT_ORDER | SDR_FIR_NO_TENSOR | SDR_FIR_NO_TCGEN05))) {
        // three bf16 terms per operand (the reference's f32 accuracy) when the tables and planes fit in shared memory
        // (K <= 384), two terms (< 1e-5 of max|y|) on request or for longer filters
        const int ns = ((flags & SDR_FIR_SPLIT2) || !fir_umma_c64_applies((int)K, (int)D, taps_complex != 0, 3)) ? 2 : 3;
        std::vector<uint8_t> tab;
        if (fir_umma_c64_applies((int)K, (int)D, taps_complex != 0, ns) && K >= 8 &&
            fir_umma_c64_build_tables(taps.data(), (int)K, ns, tab)) {
            uc_ns = ns;
            if ((rc = d_uc_tables.upload(tab.data(), tab.size(), stream.s))) return rc;
        }
    }
    return cuda_status(cudaStreamSynchronize(stream.s));
}

extern "C" sdr_fir_t *sdr_fir_create(const sdr_fir_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || cfg->n_taps == 0 || cfg->decimation == 0 || cfg->n_channels == 0 ||
        cfg->n_taps > (1u << 20) || cfg->input_format < 0 || cfg->input_format > 2 ||
        (cfg->taps_complex && cfg->input_format == SDR_FMT_F32))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_fir>(err, cfg->device, cfg->stream, [&](sdr_fir &f) {
        f.fmt = cfg->input_format;
        f.taps_complex = cfg->taps_complex ? 1 : 0;
        f.flags = cfg->flags;
        f.K = cfg->n_taps;
        f.Kp = round_up(f.K, 8);
        f.HL = f.Kp;
        f.hist_stride = f.HL;  // multiple of 8 elements: rows stay 16-byte aligned in every format
        f.D = cfg->decimation;
        f.n_ch = cfg->n_channels;
        const int w = f.taps_complex ? 2 : 1;
        f.taps.assign(f.Kp * w, 0.0f);
        std::memcpy(f.taps.data(), cfg->taps, f.K * w * sizeof(float));
        return SDR_OK;
    });
}
extern "C" void sdr_fir_destroy(sdr_fir_t *f) { destroy_handle(f); }

extern "C" int sdr_fir_reset(sdr_fir_t *f) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    DeviceGuard g(f->dev);
    if (!g.ok) return g.status();
    f->phase = 0;
    f->cur = 0;
    int rc = fir_fill_hist(f->d_hist[0].p, f->fmt, (long long)(f->n_ch * f->hist_stride), f->stream.s);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(f->stream.s));
}

extern "C" sdr_fir_t *sdr_fir_clone(const sdr_fir_t *src, int *err) { return clone_handle<FirHost>(src, err); }

extern "C" size_t sdr_fir_output_count(const sdr_fir_t *f, size_t n_in) {
    if (!f) return 0;
    const size_t first = f->D - 1 - f->phase;
    return n_in > first ? (n_in - 1 - first) / f->D + 1 : 0;
}
extern "C" int sdr_fir_last_path(const sdr_fir_t *f) { return f ? f->last_path : 0; }

static int fir_run_dev(sdr_fir *f, const void *in, size_t n_in, size_t in_stride, void *out, size_t out_stride,
                       size_t n_out) {
    FirArgs a;
    a.in = in;
    a.hist = f->d_hist[f->cur].p;
    a.out = out;
    a.taps = (const float *)f->d_taps.p;
    a.n_in = (long long)n_in;
    a.in_stride = (long long)in_stride;
    a.out_stride = (long long)out_stride;
    a.hist_stride = (long long)f->hist_stride;
    a.n_out = (long long)n_out;
    a.first = (long long)(f->D - 1 - f->phase);
    a.K = (int)f->K; a.Kp = (int)f->Kp; a.HL = (int)f->HL; a.D = (int)f->D; a.n_ch = (int)f->n_ch;
    const bool strict = (f->flags & SDR_FIR_STRICT_ORDER) != 0;
    int rc = SDR_ERR_UNSUPPORTED;
    if (f->d_um_tables.p) {
        rc = fir_umma_launch(a, f->um_R, f->um_PC, f->um_planar, (const uint8_t *)f->d_um_tables.p, f->um_magic, f->um_sc,
                             f->stream.s);
        if (rc == SDR_OK) f->last_path = 4;
    }
    if (rc == SDR_ERR_UNSUPPORTED && f->d_uc_tables.p) {
        rc = fir_umma_c64_launch(a, f->uc_ns, (const uint8_t *)f->d_uc_tables.p, f->stream.s);
        if (rc == SDR_OK) f->last_path = 5;
    }
    if (rc == SDR_ERR_UNSUPPORTED && f->d_tc_tables.p) {
        rc = fir_tc_launch(a, f->taps_complex != 0, (const uint2 *)f->d_tc_tables.p, f->tc_scale, f->stream.s);
        if (rc == SDR_OK) f->last_path = 3;
    }
    if (rc == SDR_ERR_UNSUPPORTED) rc = fir_launch(a, f->fmt, f->taps_complex != 0, strict, f->stream.s, &f->last_path);
    if (rc) return rc;
    rc = fir_hist_update(in, f->d_hist[f->cur].p, f->d_hist[f->cur ^ 1].p, f->fmt, (int)f->HL, (long long)n_in,
                         (long long)in_stride, (long long)f->hist_stride, (int)f->n_ch, f->stream.s);
    if (rc) return rc;
    f->cur ^= 1;
    f->phase = (f->phase + n_in) % f->D;
    return SDR_OK;
}

extern "C" int sdr_fir_process_dev(sdr_fir_t *f, const void *in, size_t n_in, size_t in_stride, void *out,
                                   size_t out_cap, size_t out_stride, size_t *n_used, size_t *n_out) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    if (n_used) *n_used = 0;
    if (n_out) *n_out = 0;
    if (n_in == 0) return SDR_OK;
    if (!in) return SDR_ERR_BAD_DATA_PTR;
    const size_t no = sdr_fir_output_count(f, n_in);
    if (no > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (no > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (f->n_ch == 1) { in_stride = n_in; out_stride = no; }
    if (in_stride < n_in || out_stride < no) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(f->dev);
    if (!g.ok) return g.status();
    int rc = fir_run_dev(f, in, n_in, in_stride, out, out_stride, no);
    if (rc) return rc;
    if (n_used) *n_used = n_in;
    if (n_out) *n_out = no;
    return SDR_OK;
}

extern "C" int sdr_fir_process(sdr_fir_t *f, const void *in, size_t n_in, size_t in_stride, void *out, size_t out_cap,
                               size_t out_stride, size_t *n_used, size_t *n_out) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    if (n_used) *n_used = 0;
    if (n_out) *n_out = 0;
    if (n_in == 0) return SDR_OK;
    if (!in) return SDR_ERR_BAD_DATA_PTR;
    const size_t no = sdr_fir_output_count(f, n_in);
    if (no > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (no > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (f->n_ch == 1) { in_stride = n_in; out_stride = no; }
    if (in_stride < n_in || out_stride < no) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(f->dev);
    if (!g.ok) return g.status();
    const size_t es_in = elem_bytes(f->fmt), es_out = (f->fmt == SDR_FMT_F32) ? 4 : 8;
    cudaStream_t st = f->stream.s;
    // chunks of ~32 MiB of input per channel-set, multiples of 4096*D samples so every chunk but the last keeps the
    // fast kernels' alignment and tile grid (the c64 tcgen05 kernel's 4096-output tiles then sit at the same stream
    // positions for any chunking: same bits); H2D(c+1) / kernel(c) / D2H(c-1) overlap
    size_t chunk = std::max<size_t>(1, ((size_t)32 << 20) / (es_in * f->n_ch));
    chunk = std::max<size_t>(4096 * f->D, chunk / (4096 * f->D) * (4096 * f->D));
    if (chunk > n_in) chunk = n_in;
    const size_t out_per_chunk = chunk / f->D + 2;
    const size_t ds_in = round_up(chunk, 8), ds_out = round_up(out_per_chunk, 2);
    int rc = f->pipe.init();
    DevBuf *bin[2] = {&f->d_in, &f->d_in2}, *bout[2] = {&f->d_out, &f->d_out2};
    const int nbuf = (chunk < n_in) ? 2 : 1;
    for (int i = 0; i < nbuf && !rc; ++i) {
        rc = bin[i]->reserve(f->n_ch * ds_in * es_in);
        if (!rc) rc = bout[i]->reserve(f->n_ch * ds_out * es_out);
    }
    if (rc) return rc;
    size_t done_in = 0, done_out = 0;
    for (int c = 0; done_in < n_in; ++c) {
        const int b = c & 1;
        const size_t cnt = std::min(chunk, n_in - done_in);
        const size_t cno = sdr_fir_output_count(f, cnt);
        rc = f->pipe.begin_upload(b);
        if (!rc) rc = copy2d(bin[b]->p, ds_in * es_in, (const char *)in + done_in * es_in, in_stride * es_in, cnt * es_in,
                             f->n_ch, cudaMemcpyHostToDevice, f->pipe.up);
        if (!rc) rc = f->pipe.end_upload(b);
        if (!rc) rc = f->pipe.begin_compute(b, st);
        if (!rc) rc = fir_run_dev(f, bin[b]->p, cnt, ds_in, bout[b]->p, ds_out, cno);
        if (!rc) rc = f->pipe.end_compute(b, st);
        if (!rc) rc = copy2d((char *)out + done_out * es_out, out_stride * es_out, bout[b]->p, ds_out * es_out, cno * es_out,
                             f->n_ch, cudaMemcpyDeviceToHost, f->pipe.down);
        if (!rc) rc = f->pipe.end_download(b);
        if (rc) {
            // the chunks before this one went through (their state advance is real): say so, so the caller can resume
            f->pipe.drain(st);
            if (n_used) *n_used = done_in;
            if (n_out) *n_out = done_out;
            return rc;
        }
        done_in += cnt;
        done_out += cno;
    }
    rc = f->pipe.drain(st);
    if (rc) return rc;
    if (n_used) *n_used = n_in;
    if (n_out) *n_out = done_out;
    return SDR_OK;
}

// ============================================================================================
// FFT
// ============================================================================================
struct FftHost {
    int dev = 0;
    size_t n = 0;
    int fmt = 0;
    unsigned flags = 0;
    int mode = 0;  // 0 single-launch pow2 kernels, 1 naive, 2 bluestein, 3 pow2 through convert / four-step / finish
    int log_n = 0;
    float norm = 1.0f;
    // bluestein
    size_t m = 0;
    int log_m = 0;
};

struct sdr_fft : FftHost {
    StreamRef stream;
    DevBuf d_tw;          // W_n (pow2 / naive) or W_m (bluestein), when that length is <= 2^16
    DevBuf d_tw1, d_tw2;  // lengths above 2^16: W tables of the two four-step factors
    DevBuf d_chirp, d_bfft;  // bluestein
    DevBuf d_a1, d_a2, d_work, d_h1, d_h2;
    DevBuf d_in, d_out, d_in2, d_out2;
    HostPipe pipe;

    int alloc(void *user_stream, const sdr_fft *);
};

static int upload_twiddles(DevBuf &d, size_t n, cudaStream_t st) {
    std::vector<float2> tw(n);
    const double c = -2.0 * M_PI / (double)n;
    for (size_t k = 0; k < n; ++k) tw[k] = make_float2((float)std::cos(c * (double)k), (float)std::sin(c * (double)k));
    const int rc = d.upload(tw.data(), n * sizeof(float2), st);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

static int ilog2_exact(size_t n) {
    int l = 0;
    while (((size_t)1 << l) < n) ++l;
    return (((size_t)1 << l) == n) ? l : -1;
}

constexpr int FFT_MAX_LOG = 27;  // 2^27 c64 = 1 GiB per buffer; the four-step path needs four of them

// tables for a plain c64 transform of length 2^l: one table up to 2^16, the two factor tables above
static int fft_pow2_tables(sdr_fft *p, int l) {
    cudaStream_t st = p->stream.s;
    if (l <= 16) return upload_twiddles(p->d_tw, (size_t)1 << l, st);
    const int l1 = l / 2, l2 = l - l1;
    int rc = upload_twiddles(p->d_tw1, (size_t)1 << l1, st);
    if (!rc) rc = upload_twiddles(p->d_tw2, (size_t)1 << l2, st);
    return rc;
}

// plain forward c64 -> c64 transforms of length 2^l (4 <= l <= FFT_MAX_LOG) with the plan's tables
static int fft_pow2_c64(sdr_fft *p, const float2 *in, float2 *out, int l, size_t batches) {
    cudaStream_t st = p->stream.s;
    if (l <= 16) {
        FftArgs a;
        a.in = in; a.out = out; a.tw = (const float2 *)p->d_tw.p; a.batches = (long long)batches; a.log_n = l;
        a.fmt = SDR_FMT_C64;
        a.flags = 0; a.norm = 1.0f;
        if (l >= 13) {
            const int rc = p->d_work.reserve((batches + 1) * sizeof(int));
            if (rc) return rc;
            a.work = (int *)p->d_work.p;
        }
        return fft_pow2_launch(a, st);
    }
    const size_t bytes = (batches << l) * sizeof(float2);
    int rc = p->d_h1.reserve(bytes);
    if (!rc) rc = p->d_h2.reserve(bytes);
    if (!rc) rc = p->d_work.reserve(((batches << (l - l / 2)) + 1) * sizeof(int));
    if (rc) return rc;
    return fft_huge_launch(in, out, (float2 *)p->d_h1.p, (float2 *)p->d_h2.p, (const float2 *)p->d_tw1.p,
                           (const float2 *)p->d_tw2.p, l, (long long)batches,
                           (int *)p->d_work.p, st);
}

static int fft_plan_init(sdr_fft *p) {
    cudaStream_t st = p->stream.s;
    const size_t n = p->n;
    const int l2 = ilog2_exact(n);
    if (l2 >= 4 && l2 <= 16 && !((p->flags & SDR_FFT_RFFT) && l2 >= 15)) {
        p->mode = 0;
        p->log_n = l2;
        return upload_twiddles(p->d_tw, n, st);
    }
    if (l2 >= 15) {  // 2^17 and up, and rfft of 2^15 / 2^16
        if (l2 > FFT_MAX_LOG) return SDR_ERR_UNSUPPORTED;
        p->mode = 3;
        p->log_n = l2;
        return fft_pow2_tables(p, l2);
    }
    if (n <= 64) {
        p->mode = 1;
        return upload_twiddles(p->d_tw, n, st);
    }
    // Bluestein: m = smallest power of two >= 2n-1
    p->mode = 2;
    size_t m = 16;
    while (m < 2 * n - 1) m <<= 1;
    p->m = m;
    p->log_m = ilog2_exact(m);
    if (p->log_m > FFT_MAX_LOG) return SDR_ERR_UNSUPPORTED;
    int rc = fft_pow2_tables(p, p->log_m);
    if (rc) return rc;
    std::vector<float2> chirp(n), b(m, make_float2(0.f, 0.f));
    for (size_t j = 0; j < n; ++j) {
        const unsigned long long q = ((unsigned long long)j * j) % (2ull * n);  // j^2 mod 2n keeps the angle small
        const double ang = M_PI * (double)q / (double)n;
        chirp[j] = make_float2((float)std::cos(ang), (float)-std::sin(ang));     // e^{-i pi j^2/n}
        const float2 w = make_float2((float)std::cos(ang), (float)std::sin(ang)); // e^{+i pi j^2/n}
        b[j] = w;
        if (j > 0) b[m - j] = w;
    }
    DevBuf d_b;
    if ((rc = p->d_chirp.upload(chirp.data(), n * sizeof(float2), st)) || (rc = p->d_bfft.alloc(m * sizeof(float2))) ||
        (rc = d_b.upload(b.data(), m * sizeof(float2), st)))
        return rc;
    rc = fft_pow2_c64(p, (const float2 *)d_b.p, (float2 *)p->d_bfft.p, p->log_m, 1);
    cudaError_t e = cudaStreamSynchronize(st);  // before d_b is freed
    if (rc) return rc;
    return cuda_status(e);
}

int sdr_fft::alloc(void *user_stream, const sdr_fft *) {
    int rc = stream.init(user_stream);
    return rc ? rc : fft_plan_init(this);
}

extern "C" sdr_fft_t *sdr_fft_create(const sdr_fft_config_t *cfg, int *err) {
    if (!cfg || cfg->n == 0 || cfg->input_format < 0 || cfg->input_format > 2) return fail(err, SDR_ERR_INVALID_ARG);
    if ((cfg->flags & SDR_FFT_RFFT) && cfg->input_format != SDR_FMT_F32) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_fft>(err, cfg->device, cfg->stream, [&](sdr_fft &p) {
        p.n = cfg->n;
        p.fmt = cfg->input_format;
        p.flags = cfg->flags;
        p.norm = 1.0f / sqrtf((float)cfg->n);  // fft.rs:16
        return SDR_OK;
    });
}
extern "C" void sdr_fft_destroy(sdr_fft_t *p) { destroy_handle(p); }
extern "C" size_t sdr_fft_output_len(const sdr_fft_t *p) {
    if (!p) return 0;
    return (p->flags & SDR_FFT_RFFT) ? p->n - p->n / 2 : p->n;
}

static int fft_run_dev(sdr_fft *p, const void *in, size_t batches, float *out) {
    cudaStream_t st = p->stream.s;
    if (p->mode == 0) {
        FftArgs a;
        a.in = in; a.out = (float2 *)out; a.tw = (const float2 *)p->d_tw.p; a.batches = (long long)batches; a.log_n = p->log_n;
        a.fmt = p->fmt; a.flags = p->flags; a.norm = p->norm;
        if (p->log_n >= 13) {
            const int rc = p->d_work.reserve((batches + 1) * sizeof(int));
            if (rc) return rc;
            a.work = (int *)p->d_work.p;
        }
        return fft_pow2_launch(a, st);
    }
    if (p->mode == 1)
        return fft_naive_launch(in, (float2 *)out, (const float2 *)p->d_tw.p, (long long)batches, (int)p->n, p->fmt, p->flags, p->norm, st);
    const size_t out_len = sdr_fft_output_len(p);
    if (p->mode == 3) {
        // convert -> plain c64 transform -> shift / norm / rfft selection, in slabs that bound the scratch footprint
        const size_t slab = std::max<size_t>(1, std::min<size_t>(batches, ((size_t)256 << 20) / (p->n * sizeof(float2))));
        int rc = p->d_a1.reserve(slab * p->n * sizeof(float2));
        if (!rc) rc = p->d_a2.reserve(slab * p->n * sizeof(float2));
        if (rc) return rc;
        for (size_t b0 = 0; b0 < batches; b0 += slab) {
            const size_t nb = std::min(slab, batches - b0);
            float2 *a1 = (float2 *)p->d_a1.p, *a2 = (float2 *)p->d_a2.p;
            rc = fft_convert_launch((const char *)in + b0 * p->n * elem_bytes(p->fmt), a1, (long long)(nb * p->n), p->fmt, st);
            if (!rc) rc = fft_pow2_c64(p, a1, a2, p->log_n, nb);
            if (!rc) rc = fft_finish_launch(a2, (float2 *)out + b0 * out_len, (long long)nb, (long long)p->n, p->flags, p->norm, st);
            if (rc) return rc;
        }
        return SDR_OK;
    }
    // bluestein, in slabs that bound the scratch footprint
    const size_t slab = std::max<size_t>(1, std::min<size_t>(batches, ((size_t)64 << 20) / (p->m * sizeof(float2))));
    int rc = p->d_a1.reserve(slab * p->m * sizeof(float2));
    if (!rc) rc = p->d_a2.reserve(slab * p->m * sizeof(float2));
    if (rc) return rc;
    for (size_t b0 = 0; b0 < batches; b0 += slab) {
        const size_t nb = std::min(slab, batches - b0);
        const char *inb = (const char *)in + b0 * p->n * elem_bytes(p->fmt);
        float2 *a1 = (float2 *)p->d_a1.p, *a2 = (float2 *)p->d_a2.p;
        rc = bluestein_pre_launch(inb, a1, (const float2 *)p->d_chirp.p, (long long)nb, (int)p->n, (int)p->m, p->fmt, st);
        if (rc) return rc;
        rc = fft_pow2_c64(p, a1, a2, p->log_m, nb);
        if (rc) return rc;
        rc = bluestein_mul_launch(a2, (const float2 *)p->d_bfft.p, (long long)nb, (int)p->m, st);
        if (rc) return rc;
        rc = fft_pow2_c64(p, a2, a1, p->log_m, nb);
        if (rc) return rc;
        rc = bluestein_post_launch(a1, (float2 *)out + b0 * out_len, (const float2 *)p->d_chirp.p, (long long)nb, (int)p->n, (int)p->m,
                                   p->flags, p->norm, st);
        if (rc) return rc;
    }
    return SDR_OK;
}

extern "C" int sdr_fft_exec_dev(sdr_fft_t *p, const void *in, size_t batches, float *out) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (batches == 0) return SDR_OK;
    if (!in || !out) return SDR_ERR_BAD_DATA_PTR;
    // the kernels load whole elements (u8 IQ pairs as 16-bit words) and store whole c64 values
    if (((uintptr_t)in % elem_bytes(p->fmt)) != 0 || ((uintptr_t)out % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    return fft_run_dev(p, in, batches, out);
}

extern "C" int sdr_fft_exec(sdr_fft_t *p, const void *in, size_t batches, float *out) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (batches == 0) return SDR_OK;
    if (!in || !out) return SDR_ERR_BAD_DATA_PTR;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    const size_t es = elem_bytes(p->fmt), out_len = sdr_fft_output_len(p);
    cudaStream_t st = p->stream.s;
    // chunks of ~32 MiB of input (at least one transform); H2D(c+1) / kernel(c) / D2H(c-1) overlap
    size_t chunk = std::max<size_t>(1, ((size_t)32 << 20) / (p->n * es));
    if (chunk > batches) chunk = batches;
    int rc = p->pipe.init();
    DevBuf *bin[2] = {&p->d_in, &p->d_in2}, *bout[2] = {&p->d_out, &p->d_out2};
    const int nbuf = (chunk < batches) ? 2 : 1;
    for (int i = 0; i < nbuf && !rc; ++i) {
        rc = bin[i]->reserve(chunk * p->n * es);
        if (!rc) rc = bout[i]->reserve(chunk * std::max(out_len, p->n) * sizeof(float2));
    }
    if (rc) return rc;
    size_t done = 0;
    for (int c = 0; done < batches; ++c) {
        const int b = c & 1;
        const size_t cnt = std::min(chunk, batches - done);
        rc = p->pipe.begin_upload(b);
        if (!rc) rc = cuda_status(cudaMemcpyAsync(bin[b]->p, (const char *)in + done * p->n * es, cnt * p->n * es,
                                                  cudaMemcpyHostToDevice, p->pipe.up));
        if (!rc) rc = p->pipe.end_upload(b);
        if (!rc) rc = p->pipe.begin_compute(b, st);
        if (!rc) rc = fft_run_dev(p, bin[b]->p, cnt, (float *)bout[b]->p);
        if (!rc) rc = p->pipe.end_compute(b, st);
        if (!rc) rc = cuda_status(cudaMemcpyAsync((char *)out + done * out_len * sizeof(float2), bout[b]->p,
                                                  cnt * out_len * sizeof(float2), cudaMemcpyDeviceToHost, p->pipe.down));
        if (!rc) rc = p->pipe.end_download(b);
        if (rc) { p->pipe.drain(st); return rc; }
        done += cnt;
    }
    return p->pipe.drain(st);
}

// fft.rs:14-24: fstep = rate / (len as f32); start = -(len as isize / 2); label = srci as f32 * fstep
extern "C" int sdr_fft_labels(size_t n, float rate, int rfft, float *labels) {
    if (n == 0) return SDR_OK;
    if (!labels) return SDR_ERR_BAD_DATA_PTR;
    const float fstep = rate / (float)n;
    const long start = -((long)n / 2);
    const size_t drop = rfft ? n / 2 : 0;
    for (size_t i = drop; i < n; ++i) labels[i - drop] = (float)(start + (long)i) * fstep;
    return SDR_OK;
}

// ============================================================================================
// Biquad design + PLL
// ============================================================================================
// biquad.rs:83-154 (design, f32 throughout) and :25-38 (division by a0)
extern "C" int sdr_biquad_design(const sdr_biquad_design_t *d, float rate, float coef[5]) {
    if (!d || !coef) return SDR_ERR_BAD_DATA_PTR;
    const float PI_F = 3.14159265358979323846f;
    float a0 = 1, a1 = 0, a2 = 0, b0 = 1, b1 = 0, b2 = 0;
    switch (d->kind) {
        case SDR_BQ_IDENTITY: break;
        case SDR_BQ_LOWPASS: case SDR_BQ_HIGHPASS: case SDR_BQ_BANDPASS: case SDR_BQ_NOTCH: {
            const float omega = 2.0f * PI_F * d->p0 / rate;
            const float cs = cosf(omega);
            const float alpha = sinf(omega) / (2.0f * d->p1);
            a0 = 1.0f + alpha; a1 = -2.0f * cs; a2 = 1.0f - alpha;
            if (d->kind == SDR_BQ_LOWPASS) { b0 = (1.0f - cs) / 2.0f; b1 = 1.0f - cs; b2 = (1.0f - cs) / 2.0f; }
            else if (d->kind == SDR_BQ_HIGHPASS) { b0 = (1.0f + cs) / 2.0f; b1 = -1.0f - cs; b2 = (1.0f + cs) / 2.0f; }
            else if (d->kind == SDR_BQ_BANDPASS) { b0 = alpha; b1 = 0.0f; b2 = -alpha; }
            else { b0 = 1.0f; b1 = -2.0f * cs; b2 = 1.0f; }
            break;
        }
        case SDR_BQ_LR: {
            const float decayn = d->p0 / rate;
            a0 = 1.0f; a1 = -expf(-decayn); a2 = 0.0f; b0 = decayn; b1 = 0.0f; b2 = 0.0f;
            break;
        }
        default: return SDR_ERR_INVALID_ARG;
    }
    coef[0] = b0 / a0; coef[1] = b1 / a0; coef[2] = b2 / a0; coef[3] = -a1 / a0; coef[4] = -a2 / a0;
    return SDR_OK;
}

struct PllHost {
    int dev = 0;
    size_t n_streams = 0, n_designs = 0;
    unsigned flags = 0;
    std::vector<PllParams> params;
    bool any_identity = false;  // some sub-filter is filter::Identity: the kernel keeps its per-filter kind tests
};

struct sdr_pll : PllHost {
    StreamRef stream;
    DevBuf d_params, d_state;
    DevBuf d_in, d_out, d_lk;

    int alloc(void *user_stream, const sdr_pll *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_params.upload(params.data(), params.size() * sizeof(PllParams), stream.s)) ||
            (rc = d_state.alloc(n_streams * sizeof(PllState))))
            return rc;
        SDR_CUDA_TRY(cudaMemsetAsync(d_state.p, 0, n_streams * sizeof(PllState), stream.s));  // pll.rs:57-58
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_pll &src) {
        return cuda_status(cudaMemcpy(d_state.p, src.d_state.p, n_streams * sizeof(PllState), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_pll_t *sdr_pll_create(const sdr_pll_config_t *cfg, int *err) {
    if (!cfg || !cfg->designs || cfg->n_streams == 0 || cfg->n_streams > (1u << 24) ||
        (cfg->n_designs != 1 && cfg->n_designs != cfg->n_streams))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_pll>(err, cfg->device, cfg->stream, [&](sdr_pll &p) {
        p.n_streams = cfg->n_streams;
        p.n_designs = cfg->n_designs;
        p.flags = cfg->flags;
        p.params.resize(cfg->n_designs);
        for (size_t i = 0; i < cfg->n_designs; ++i) {
            const sdr_pll_design_t &d = cfg->designs[i];
            PllParams &q = p.params[i];
            q.reference = d.reference / cfg->rate;  // pll.rs:51
            q.gain = d.gain;
            q.rate = cfg->rate;
            q.lk = d.loopfilter.kind; q.ok = d.outputfilter.kind; q.kk = d.lockfilter.kind;
            if (q.lk == SDR_BQ_IDENTITY || q.ok == SDR_BQ_IDENTITY || q.kk == SDR_BQ_IDENTITY) p.any_identity = true;
            // the specialised kernel also assumes |nphase + reference + gain * arg| < 2 (nphase in (-1, 1), |arg| <= pi), so
            // that f32::fract needs no general trunc; designs with a larger step per sample take the general kernel
            if (!(std::fabs(q.reference) + 3.1416f * std::fabs(q.gain) < 0.999f)) p.any_identity = true;
            if (cfg->flags & SDR_PLL_GENERAL_KERNEL) p.any_identity = true;
            int rc = sdr_biquad_design(&d.loopfilter, cfg->rate, q.lc);
            if (!rc) rc = sdr_biquad_design(&d.outputfilter, cfg->rate, q.oc);
            if (!rc) rc = sdr_biquad_design(&d.lockfilter, cfg->rate, q.kc);
            if (rc) return rc;
        }
        return SDR_OK;
    });
}
extern "C" void sdr_pll_destroy(sdr_pll_t *p) { destroy_handle(p); }
extern "C" int sdr_pll_reset(sdr_pll_t *p) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    SDR_CUDA_TRY(cudaMemsetAsync(p->d_state.p, 0, p->n_streams * sizeof(PllState), p->stream.s));
    return cuda_status(cudaStreamSynchronize(p->stream.s));
}
extern "C" sdr_pll_t *sdr_pll_clone(const sdr_pll_t *src, int *err) { return clone_handle<PllHost>(src, err); }

extern "C" int sdr_pll_process_dev(sdr_pll_t *p, const float *in, size_t n, size_t in_stride, float *out,
                                   uint8_t *locked, size_t out_stride) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out || !locked) return SDR_ERR_BAD_DATA_PTR;
    if (p->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    return pll_launch((const float2 *)in, (long long)n, (long long)in_stride, out, locked, (long long)out_stride,
                      (const PllParams *)p->d_params.p, p->n_designs == 1, (PllState *)p->d_state.p, (int)p->n_streams,
                      (p->flags & SDR_PLL_F64_MATH) == 0, p->any_identity, p->stream.s);
}

extern "C" int sdr_pll_process(sdr_pll_t *p, const float *in, size_t n, size_t in_stride, float *out, uint8_t *locked,
                               size_t out_stride) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out || !locked) return SDR_ERR_BAD_DATA_PTR;
    if (p->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    const size_t S = p->n_streams;
    int rc = p->d_in.reserve(S * n * 8);
    if (!rc) rc = p->d_out.reserve(S * n * 4);
    if (!rc) rc = p->d_lk.reserve(S * n);
    if (rc) return rc;
    cudaStream_t st = p->stream.s;
    rc = copy2d(p->d_in.p, n * 8, in, in_stride * 8, n * 8, S, cudaMemcpyHostToDevice, st);
    if (rc) return rc;
    rc = pll_launch((const float2 *)p->d_in.p, (long long)n, (long long)n, (float *)p->d_out.p, (uint8_t *)p->d_lk.p,
                    (long long)n, (const PllParams *)p->d_params.p, p->n_designs == 1, (PllState *)p->d_state.p, (int)S,
                    (p->flags & SDR_PLL_F64_MATH) == 0, p->any_identity, st);
    if (rc) return rc;
    rc = copy2d(out, out_stride * 4, p->d_out.p, n * 4, n * 4, S, cudaMemcpyDeviceToHost, st);
    if (!rc) rc = copy2d(locked, out_stride, p->d_lk.p, n, n, S, cudaMemcpyDeviceToHost, st);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

extern "C" int sdr_pll_stereo_decode_dev(sdr_pll_t *p, const float *v, size_t n, size_t in_stride, float *out_md,
                                         size_t out_stride) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!v || !out_md) return SDR_ERR_BAD_DATA_PTR;
    if (p->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    return pll_stereo_launch(v, (long long)n, (long long)in_stride, out_md, (long long)out_stride,
                             (const PllParams *)p->d_params.p, p->n_designs == 1, (PllState *)p->d_state.p,
                             (int)p->n_streams, (p->flags & SDR_PLL_F64_MATH) == 0, p->stream.s);
}

extern "C" int sdr_pll_stereo_decode(sdr_pll_t *p, const float *v, size_t n, size_t in_stride, float *out_md,
                                     size_t out_stride) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!v || !out_md) return SDR_ERR_BAD_DATA_PTR;
    if (p->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    const size_t S = p->n_streams;
    int rc = p->d_in.reserve(S * n * 4);
    if (!rc) rc = p->d_out.reserve(S * n * 8);
    if (rc) return rc;
    cudaStream_t st = p->stream.s;
    rc = copy2d(p->d_in.p, n * 4, v, in_stride * 4, n * 4, S, cudaMemcpyHostToDevice, st);
    if (rc) return rc;
    rc = pll_stereo_launch((const float *)p->d_in.p, (long long)n, (long long)n, (float *)p->d_out.p, (long long)n,
                           (const PllParams *)p->d_params.p, p->n_designs == 1, (PllState *)p->d_state.p, (int)S,
                           (p->flags & SDR_PLL_F64_MATH) == 0, st);
    if (rc) return rc;
    rc = copy2d(out_md, out_stride * 8, p->d_out.p, n * 8, n * 8, S, cudaMemcpyDeviceToHost, st);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

extern "C" int sdr_pll_get_state(sdr_pll_t *p, size_t idx, float *nphase, float *vre, float *vim) {
    if (!p) return SDR_ERR_NULL_HANDLE;
    if (idx >= p->n_streams) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(p->dev);
    if (!g.ok) return g.status();
    PllState s;
    SDR_CUDA_TRY(cudaStreamSynchronize(p->stream.s));
    SDR_CUDA_TRY(cudaMemcpy(&s, (const PllState *)p->d_state.p + idx, sizeof(s), cudaMemcpyDeviceToHost));
    if (nphase) *nphase = s.nphase;
    if (vre) *vre = s.vre;
    if (vim) *vim = s.vim;
    return SDR_OK;
}

// ============================================================================================
// Biquad stream filter
// ============================================================================================
struct BiquadHost {
    int dev = 0;
    size_t n_streams = 0, n_designs = 0;
    int W = 1;
    std::vector<float> coef;  // 5 per design
    std::vector<int> kind;
};

struct sdr_biquad : BiquadHost {
    StreamRef stream;
    DevBuf d_coef, d_kind, d_state;
    DevBuf d_in, d_out;

    size_t state_bytes() const { return n_streams * W * 4 * sizeof(float); }
    int alloc(void *user_stream, const sdr_biquad *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_coef.upload(coef.data(), coef.size() * sizeof(float), stream.s)) ||
            (rc = d_kind.upload(kind.data(), kind.size() * sizeof(int), stream.s)) || (rc = d_state.alloc(state_bytes())))
            return rc;
        SDR_CUDA_TRY(cudaMemsetAsync(d_state.p, 0, state_bytes(), stream.s));
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_biquad &src) {
        return cuda_status(cudaMemcpy(d_state.p, src.d_state.p, state_bytes(), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_biquad_t *sdr_biquad_create(const sdr_biquad_config_t *cfg, int *err) {
    if (!cfg || !cfg->designs || cfg->n_streams == 0 || cfg->n_streams > (1u << 24) ||
        (cfg->n_designs != 1 && cfg->n_designs != cfg->n_streams))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_biquad>(err, cfg->device, cfg->stream, [&](sdr_biquad &b) {
        b.n_streams = cfg->n_streams;
        b.n_designs = cfg->n_designs;
        b.W = cfg->sample_complex ? 2 : 1;
        b.coef.resize(5 * cfg->n_designs);
        b.kind.resize(cfg->n_designs);
        for (size_t i = 0; i < cfg->n_designs; ++i) {
            b.kind[i] = cfg->designs[i].kind;
            const int rc = sdr_biquad_design(&cfg->designs[i], cfg->rate, &b.coef[5 * i]);
            if (rc) return rc;
        }
        return SDR_OK;
    });
}
extern "C" void sdr_biquad_destroy(sdr_biquad_t *b) { destroy_handle(b); }
extern "C" int sdr_biquad_reset(sdr_biquad_t *b) {
    if (!b) return SDR_ERR_NULL_HANDLE;
    DeviceGuard g(b->dev);
    if (!g.ok) return g.status();
    SDR_CUDA_TRY(cudaMemsetAsync(b->d_state.p, 0, b->state_bytes(), b->stream.s));
    return cuda_status(cudaStreamSynchronize(b->stream.s));
}
extern "C" sdr_biquad_t *sdr_biquad_clone(const sdr_biquad_t *src, int *err) { return clone_handle<BiquadHost>(src, err); }
extern "C" int sdr_biquad_process_dev(sdr_biquad_t *b, const float *in, size_t n, size_t in_stride, float *out, size_t out_stride) {
    if (!b) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out) return SDR_ERR_BAD_DATA_PTR;
    if (b->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(b->dev);
    if (!g.ok) return g.status();
    return biquad_launch(in, (long long)n, (long long)in_stride, out, (long long)out_stride, b->W,
                         (const float *)b->d_coef.p, (const int *)b->d_kind.p, b->n_designs == 1, (float *)b->d_state.p,
                         (int)(b->n_streams * b->W), b->stream.s);
}
extern "C" int sdr_biquad_process(sdr_biquad_t *b, const float *in, size_t n, size_t in_stride, float *out, size_t out_stride) {
    if (!b) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out) return SDR_ERR_BAD_DATA_PTR;
    if (b->n_streams == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(b->dev);
    if (!g.ok) return g.status();
    const size_t S = b->n_streams, eb = 4 * (size_t)b->W;
    int rc = b->d_in.reserve(S * n * eb);
    if (!rc) rc = b->d_out.reserve(S * n * eb);
    if (rc) return rc;
    cudaStream_t st = b->stream.s;
    rc = copy2d(b->d_in.p, n * eb, in, in_stride * eb, n * eb, S, cudaMemcpyHostToDevice, st);
    if (!rc)
        rc = biquad_launch((const float *)b->d_in.p, (long long)n, (long long)n, (float *)b->d_out.p, (long long)n, b->W,
                           (const float *)b->d_coef.p, (const int *)b->d_kind.p, b->n_designs == 1, (float *)b->d_state.p,
                           (int)(S * b->W), st);
    if (!rc) rc = copy2d(out, out_stride * eb, b->d_out.p, n * eb, n * eb, S, cudaMemcpyDeviceToHost, st);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

// ============================================================================================
// channelizer: n_channels x (FIR -> PLL).  The FIR output is produced in L2-sized slabs that the
// PLL kernel consumes immediately on the same stream.
// ============================================================================================
struct sdr_channelizer {
    Owned<sdr_fir, sdr_fir_destroy> fir;
    Owned<sdr_pll, sdr_pll_destroy> pll;
    DevBuf mid;
    DevBuf d_in, d_out, d_lk;
};

extern "C" sdr_channelizer_t *sdr_channelizer_create(const sdr_fir_config_t *fc, const sdr_pll_config_t *pc, int *err) {
    if (!fc || !pc || fc->n_channels != pc->n_streams || fc->decimation != 1 || fc->input_format == SDR_FMT_F32 ||
        fc->device != pc->device)
        return fail(err, SDR_ERR_INVALID_ARG);
    sdr_channelizer *c = new (std::nothrow) sdr_channelizer;
    if (!c) return fail(err, SDR_ERR_MALLOC_FAILED);
    c->fir.reset(sdr_fir_create(fc, err));
    if (c->fir) {
        sdr_pll_config_t pc2 = *pc;
        pc2.stream = (void *)c->fir->stream.s;  // one stream: FIR slab i is followed by PLL slab i
        c->pll.reset(sdr_pll_create(&pc2, err));
    }
    if (c->pll) return c;
    delete c;
    return nullptr;
}
extern "C" void sdr_channelizer_destroy(sdr_channelizer_t *c) {
    if (!c) return;
    DeviceGuard g(c->fir->dev);
    delete c;
}
extern "C" int sdr_channelizer_reset(sdr_channelizer_t *c) {
    if (!c) return SDR_ERR_NULL_HANDLE;
    int rc = sdr_fir_reset(c->fir.get());
    if (!rc) rc = sdr_pll_reset(c->pll.get());
    return rc;
}

extern "C" int sdr_channelizer_process_dev(sdr_channelizer_t *c, const void *in, size_t n, size_t in_stride, float *out,
                                           uint8_t *locked, size_t out_stride) {
    if (!c) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out || !locked) return SDR_ERR_BAD_DATA_PTR;
    const size_t C = c->fir->n_ch;
    if (C == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(c->fir->dev);
    if (!g.ok) return g.status();
    // slab: keep the c64 intermediate around 32 MiB so it lives in the 126 MB L2; a multiple of the FIR kernel's
    // 4096-output tile, so a channel's samples meet the same tile grid however many channels share the handle
    size_t slab = std::max<size_t>(4096, (((size_t)32 << 20) / (8 * C)) / 4096 * 4096);
    slab = std::min(slab, round_up(n, 8));
    int rc = c->mid.reserve(C * slab * 8);
    if (rc) return rc;
    const size_t es = elem_bytes(c->fir->fmt);
    for (size_t s0 = 0; s0 < n; s0 += slab) {
        const size_t cnt = std::min(slab, n - s0);
        size_t used = 0, got = 0;
        rc = sdr_fir_process_dev(c->fir.get(), (const char *)in + s0 * es, cnt, in_stride, c->mid.p, slab, slab, &used, &got);
        if (rc) return rc;
        if (C == 1) {
            rc = sdr_pll_process_dev(c->pll.get(), (const float *)c->mid.p, cnt, cnt, out + s0, locked + s0, cnt);
        } else {
            rc = sdr_pll_process_dev(c->pll.get(), (const float *)c->mid.p, cnt, slab, out + s0, locked + s0, out_stride);
        }
        if (rc) return rc;
    }
    return SDR_OK;
}

extern "C" int sdr_channelizer_process(sdr_channelizer_t *c, const void *in, size_t n, size_t in_stride, float *out,
                                       uint8_t *locked, size_t out_stride) {
    if (!c) return SDR_ERR_NULL_HANDLE;
    if (n == 0) return SDR_OK;
    if (!in || !out || !locked) return SDR_ERR_BAD_DATA_PTR;
    const size_t C = c->fir->n_ch;
    if (C == 1) { in_stride = n; out_stride = n; }
    if (in_stride < n || out_stride < n) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(c->fir->dev);
    if (!g.ok) return g.status();
    const size_t es = elem_bytes(c->fir->fmt);
    const size_t ds = round_up(n, 8);
    int rc = c->d_in.reserve(C * ds * es);
    if (!rc) rc = c->d_out.reserve(C * ds * 4);
    if (!rc) rc = c->d_lk.reserve(C * ds);
    if (rc) return rc;
    cudaStream_t st = c->fir->stream.s;
    rc = copy2d(c->d_in.p, ds * es, in, in_stride * es, n * es, C, cudaMemcpyHostToDevice, st);
    if (rc) return rc;
    rc = sdr_channelizer_process_dev(c, c->d_in.p, n, ds, (float *)c->d_out.p, (uint8_t *)c->d_lk.p, ds);
    if (rc) return rc;
    rc = copy2d(out, out_stride * 4, c->d_out.p, ds * 4, n * 4, C, cudaMemcpyDeviceToHost, st);
    if (!rc) rc = copy2d(locked, out_stride, c->d_lk.p, ds, n, C, cudaMemcpyDeviceToHost, st);
    if (rc) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

// ============================================================================================
// resampler ("sdr-src": see DESIGN.md).  Host side = the position/count state machine; the device
// holds the carried frames followed by the current input in one contiguous buffer v.
// ============================================================================================
struct SrcHost {
    int dev = 0;
    int type = 0, channels = 1;
    double ratio = 0.0;
    bool fresh = true;
    // ZOH / linear: pos relative to in[0]; one carried frame (frame -1)
    double pos = -1.0;
    // sinc: position relative to v[0]; `kept` carried frames; totals for the end-of-input rule
    double spos = 0.0;
    long long kept = 0, total_in = 0, origin_abs = 0;
    bool ended = false;
    bool exact = false;  // sdr_src_set_exact: always take the f64 kernels
};

struct sdr_src : SrcHost {
    StreamRef stream;
    DevBuf d_table;
    DevBuf v[2];
    int cur = 0;
    DevBuf carry;  // ZOH / linear: the frame before in[0]
    DevBuf d_out;
    DevBuf coef;   // sinc: per-phase wing coefficients of the polyphase fast path
    // tensor-core path (integer step, 2 channels), built on first use: branch filters' Toeplitz tables, phase planes
    int fast_S = 0, fast_Kb = 0, fast_ns = 0;
    double fast_ratio = 0.0;
    DevBuf d_fast_tab; // [S][2 deltas][KS][(32 ns) x 32 B]
    size_t fast_tab_stride = 0;
    DevBuf fast_planes;

    int alloc(void *user_stream, const sdr_src *) {
        int rc = stream.init(user_stream);
        if (rc || type > SDR_SRC_SINC_FASTEST) return rc;
        const float *tab = nullptr;
        int inc = 0;
        const size_t hl = src_sinc_table_host(type, &tab, &inc);
        return d_table.upload(tab, (hl + 2) * sizeof(float), stream.s);
    }
    int copy_device(const sdr_src &o) {
        const bool zl = type >= SDR_SRC_ZERO_ORDER_HOLD;
        const size_t bytes = (size_t)(zl ? 1 : kept) * channels * sizeof(float);
        DevBuf &dst = zl ? carry : v[0];
        const DevBuf &from = zl ? o.carry : o.v[o.cur];
        int rc = dst.reserve(std::max<size_t>(bytes, 16));
        if (!rc && bytes && from.p) rc = cuda_status(cudaMemcpy(dst.p, from.p, bytes, cudaMemcpyDeviceToDevice));
        return rc;
    }
};

static bool bad_ratio(double r) { return !(r >= 1.0 / 256.0 && r <= 256.0); }

static void src_reset_state(sdr_src *s) {
    s->ratio = 0.0; s->fresh = true; s->pos = -1.0; s->spos = 0.0; s->kept = 0; s->total_in = 0; s->origin_abs = 0;
    s->ended = false; s->cur = 0;
}

extern "C" SDR_SRC_STATE *sdr_src_new_on(int type, int channels, int device, void *stream, int *error) {
    if (channels < 1) return fail(error, SDR_ERR_BAD_CHANNEL_COUNT);
    if (type < 0 || type > 4) return fail(error, SDR_ERR_BAD_CONVERTER);
    return create_handle<sdr_src>(error, device, stream, [&](sdr_src &s) {
        s.type = type;
        s.channels = channels;
        return SDR_OK;
    });
}
extern "C" SDR_SRC_STATE *sdr_src_new(int type, int channels, int *error) {
    return sdr_src_new_on(type, channels, 0, nullptr, error);
}
extern "C" SDR_SRC_STATE *sdr_src_delete(SDR_SRC_STATE *s) {
    destroy_handle(s);
    return nullptr;
}
extern "C" int sdr_src_reset(SDR_SRC_STATE *s) {
    if (!s) return SDR_ERR_BAD_STATE;
    src_reset_state(s);
    return SDR_OK;
}
extern "C" int sdr_src_set_ratio(SDR_SRC_STATE *s, double r) {
    if (!s) return SDR_ERR_BAD_STATE;
    if (bad_ratio(r)) return SDR_ERR_BAD_SRC_RATIO;
    s->ratio = r;
    return SDR_OK;
}
extern "C" int sdr_src_get_channels(SDR_SRC_STATE *s) { return s ? s->channels : -SDR_ERR_BAD_STATE; }
extern "C" int sdr_src_set_exact(SDR_SRC_STATE *s, int exact) {
    if (!s) return SDR_ERR_BAD_STATE;
    s->exact = exact != 0;
    return SDR_OK;
}
extern "C" long sdr_src_history_frames(SDR_SRC_STATE *s) {
    if (!s) return -SDR_ERR_BAD_STATE;
    return s->type >= SDR_SRC_ZERO_ORDER_HOLD ? (s->fresh ? 0 : 1) : (long)s->kept;
}
extern "C" const char *sdr_src_strerror(int e) {
    if (e < 0 || (e > 22 && e < 100)) return nullptr;
    return sdr_strerror(e);
}
extern "C" const char *sdr_src_get_name(int t) {
    switch (t) {
        case SDR_SRC_SINC_BEST_QUALITY: return "Best Sinc Interpolator";
        case SDR_SRC_SINC_MEDIUM_QUALITY: return "Medium Sinc Interpolator";
        case SDR_SRC_SINC_FASTEST: return "Fastest Sinc Interpolator";
        case SDR_SRC_ZERO_ORDER_HOLD: return "ZOH Interpolator";
        case SDR_SRC_LINEAR: return "Linear Interpolator";
    }
    return nullptr;
}
extern "C" const char *sdr_src_get_description(int t) {
    switch (t) {
        case SDR_SRC_SINC_BEST_QUALITY: return "Band limited sinc interpolation, best quality, ~145dB SNR, 93% BW (sdr-src, B200).";
        case SDR_SRC_SINC_MEDIUM_QUALITY: return "Band limited sinc interpolation, medium quality, ~97dB SNR, 86% BW (sdr-src, B200).";
        case SDR_SRC_SINC_FASTEST: return "Band limited sinc interpolation, fastest, ~97dB SNR, 68% BW (sdr-src, B200).";
        case SDR_SRC_ZERO_ORDER_HOLD: return "Zero order hold interpolator, very fast, poor quality.";
        case SDR_SRC_LINEAR: return "Linear interpolator, very fast, poor quality.";
    }
    return nullptr;
}
extern "C" const char *sdr_src_get_version(void) { return "sdr-src-b200 1.0 (libsamplerate-shaped API, CUDA sm_100a)"; }
extern "C" size_t sdr_src_sinc_table(int type, const float **table, int *increment) {
    return src_sinc_table_host(type, table, increment);
}

extern "C" SDR_SRC_STATE *sdr_src_clone(SDR_SRC_STATE *o, int *error) {
    if (!o) return fail(error, SDR_ERR_BAD_STATE);
    return clone_handle<SrcHost>(o, error);
}

// number of outputs m in [0, cap] such that ok(m') holds for all m' < m, where ok is monotone
template <class F>
static long long count_outputs(long long cap, F &&ok) {
    long long lo = 0, hi = cap;  // invariant: ok(m) for m < lo ; !ok(m) for m >= hi (or hi == cap)
    while (lo < hi) {
        const long long mid = lo + (hi - lo) / 2;
        if (ok(mid)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Long calls at an integer step (ratio 1/S: the reference's 240 k -> 48 k and 144 k -> 48 k conversions) on a c64 stream:
// the sinc converter IS a polyphase decimating FIR with fixed taps, and runs as S branch filters on the tcgen05 Toeplitz
// kernel (fir_umma_c64.cu) instead of 2 wc f64 multiply-adds per output on the 64-lane f64 pipe.  f32 accumulation of
// bf16-split operands: within 1e-5 of max|y| of the f64 specification (north star tolerance for "resample"; measured
// ~1e-6); sdr_src_set_exact(state, 1) keeps the f64 kernels (equal to the specification up to the final f32 rounding).
constexpr long long SRC_FAST_MIN_OUT = 8192;
static int src_fast_run(sdr_src *s, const SrcLaunch &L, cudaStream_t st) {
    if (L.channels != 2 || L.type > SDR_SRC_SINC_FASTEST || L.origin != 0) return SDR_ERR_UNSUPPORTED;
    const double step = L.step;
    const long long S = (long long)step;
    if ((double)S != step || S < 1 || S > 64) return SDR_ERR_UNSUPPORTED;
    const long long P = (long long)L.pos;
    if ((double)P != L.pos || P < 0) return SDR_ERR_UNSUPPORTED;
    if (((uintptr_t)L.out & 15) || ((uintptr_t)L.v & 7)) return SDR_ERR_UNSUPPORTED;
    const int Kb = src_fast_branch_len(L.wc, (int)S);
    const int ns = fir_umma_c64_applies(Kb, 1, false, 3) ? 3 : 2;
    if (!fir_umma_c64_applies(Kb, 1, false, ns)) return SDR_ERR_UNSUPPORTED;
    const double ratio = 1.0 / step;
    if (!s->d_fast_tab.p || s->fast_S != (int)S || s->fast_Kb != Kb || s->fast_ns != ns || s->fast_ratio != ratio) {
        // (re)build the branch filters' Toeplitz tables: once per (converter, ratio), reused by every later call
        std::vector<float> br;
        src_fast_taps(s->type, ratio, (int)S, br);
        std::vector<uint8_t> all, one;
        for (long long b = 0; b < S; ++b) {
            if (!fir_umma_c64_build_tables(br.data() + (size_t)b * Kb, Kb, ns, one)) return SDR_ERR_UNSUPPORTED;
            all.insert(all.end(), one.begin(), one.end());
        }
        if (s->d_fast_tab.p) cudaStreamSynchronize(st);  // the old tables may still be in use
        int rc = s->d_fast_tab.upload(all.data(), all.size(), st);
        if (rc) return rc;
        SDR_CUDA_TRY(cudaStreamSynchronize(st));  // `all` is pageable host memory
        s->fast_tab_stride = one.size();
        s->fast_S = (int)S; s->fast_Kb = Kb; s->fast_ns = ns; s->fast_ratio = ratio;
    }
    const long long opitch = (L.n_out + 7) & ~7LL;           // branch outputs (S > 1): rows of opitch frames
    int rc = SDR_OK;
    float *bout = nullptr;
    if (S > 1) {
        rc = s->fast_planes.reserve((size_t)S * opitch * sizeof(float2));
        if (rc) return rc;
        bout = (float *)s->fast_planes.p;
    }
    // ONE launch: the S phase planes are S "channels" with their own taps, gathered by the kernel's producers straight from
    // the handle's frames (x_s[u] = v[S u + P + W - s]); every CTA is bound to one branch (one table in shared memory) and
    // the S * ceil(n_out / 4096) tiles spread over the SMs (11 waves for C3 instead of 5 launches x 3)
    FirArgs a;
    a.in = L.v;
    a.hist = L.v;
    a.out = S > 1 ? bout : L.out;
    a.taps = nullptr;
    a.n_in = L.n_out; a.in_stride = 0; a.out_stride = opitch; a.hist_stride = 0; a.n_out = L.n_out;
    a.first = 0;
    a.K = Kb; a.Kp = Kb; a.HL = 0; a.D = 1; a.n_ch = (int)S;
    a.in_step = S; a.in_off = P + L.wc + 1; a.in_limit = L.have;
    rc = fir_umma_c64_launch(a, ns, (const uint8_t *)s->d_fast_tab.p, st, S > 1 ? (long long)s->fast_tab_stride : 0);
    if (rc) return rc;
    if (S > 1) rc = src_fast_sum(bout, opitch, (int)S, L.out, L.n_out, st);
    return rc;
}

static int src_process_impl(sdr_src *s, SDR_SRC_DATA *d, bool dev_ptrs) {
    if (!s) return SDR_ERR_BAD_STATE;
    if (!d) return SDR_ERR_BAD_DATA;
    if ((d->data_in == nullptr && d->input_frames > 0) || (d->data_out == nullptr && d->output_frames > 0))
        return SDR_ERR_BAD_DATA_PTR;
    if (bad_ratio(d->src_ratio)) return SDR_ERR_BAD_SRC_RATIO;
    if (d->input_frames < 0) d->input_frames = 0;
    if (d->output_frames < 0) d->output_frames = 0;
    d->input_frames_used = 0;
    d->output_frames_gen = 0;
    s->ratio = d->src_ratio;
    const int ch = s->channels;
    const long long n = d->input_frames, cap = d->output_frames;
    const double step = 1.0 / s->ratio;
    DeviceGuard g(s->dev);
    if (!g.ok) return g.status();
    cudaStream_t st = s->stream.s;
    const cudaMemcpyKind kin = dev_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const size_t fb = (size_t)ch * sizeof(float);  // bytes per frame

    SrcLaunch L;
    L.channels = ch; L.type = s->type; L.step = step;
    L.table = (const float *)s->d_table.p; L.half_len = 0; L.rq = 0; L.rho = 0; L.wc = 0;
    long long m = 0;

    if (s->type >= SDR_SRC_ZERO_ORDER_HOLD) {
        if (n <= 0) return SDR_OK;
        DevBuf &V = s->v[s->cur];
        int rc = V.reserve((size_t)(n + 1) * fb);
        if (rc) return rc;
        DevBuf &C = s->carry;
        rc = C.reserve(fb);
        if (rc) return rc;
        if (s->fresh) {  // libsamplerate: the frame before the first is the first frame itself
            SDR_CUDA_TRY(cudaMemcpyAsync(C.p, d->data_in, fb, kin, st));
            s->fresh = false;
        }
        SDR_CUDA_TRY(cudaMemcpyAsync(V.p, C.p, fb, cudaMemcpyDeviceToDevice, st));
        SDR_CUDA_TRY(cudaMemcpyAsync((char *)V.p + fb, d->data_in, (size_t)n * fb, kin, st));
        const double P = s->pos;
        const bool lin = (s->type == SDR_SRC_LINEAR);
        m = count_outputs(cap, [&](long long mm) {
            const double Pm = P + (double)mm * step;
            return lin ? (Pm < (double)(n - 1)) : (Pm <= (double)(n - 1));
        });
        L.v = (const float *)V.p; L.have = n + 1; L.origin = 1; L.pos = P; L.n_out = m;
        const double Pn = P + (double)m * step;
        long long used = std::min<long long>((long long)std::floor(Pn) + 1, n);
        if (used < 0) used = 0;
        // outputs
        float *dout = d->data_out;
        if (!dev_ptrs) {
            rc = s->d_out.reserve(std::max<size_t>((size_t)m * fb, 16));
            if (rc) return rc;
            dout = (float *)s->d_out.p;
        }
        L.out = dout;
        rc = src_launch(L, st);
        if (rc) return rc;
        if (!dev_ptrs && m > 0) SDR_CUDA_TRY(cudaMemcpyAsync(d->data_out, dout, (size_t)m * fb, cudaMemcpyDeviceToHost, st));
        if (used > 0) SDR_CUDA_TRY(cudaMemcpyAsync(C.p, (char *)V.p + (size_t)used * fb, fb, cudaMemcpyDeviceToDevice, st));
        s->pos = Pn - (double)used;
        d->input_frames_used = (long)used;
        d->output_frames_gen = (long)m;
        if (!dev_ptrs) SDR_CUDA_TRY(cudaStreamSynchronize(st));
        return SDR_OK;
    }

    // ---- sinc ----
    double rq, rho;
    long long wc;
    src_sinc_wing(s->type, s->ratio, &rq, &rho, &wc);
    const float *tab_host = nullptr;
    int inc = 0;
    const long long half_len = (long long)src_sinc_table_host(s->type, &tab_host, &inc);
    const long long have = s->kept + n;
    DevBuf &V = s->v[s->cur];
    DevBuf &W = s->v[s->cur ^ 1];
    int rc = SDR_OK;
    if (V.cap < (size_t)std::max<long long>(have, 1) * fb) {
        // grow, preserving the carried frames
        rc = W.reserve((size_t)std::max<long long>(have, 1) * fb);
        if (rc) return rc;
        if (s->kept > 0) SDR_CUDA_TRY(cudaMemcpyAsync(W.p, V.p, (size_t)s->kept * fb, cudaMemcpyDeviceToDevice, st));
        s->cur ^= 1;
    }
    DevBuf &V2 = s->v[s->cur];
    DevBuf &W2 = s->v[s->cur ^ 1];
    if (n > 0) SDR_CUDA_TRY(cudaMemcpyAsync((char *)V2.p + (size_t)s->kept * fb, d->data_in, (size_t)n * fb, kin, st));
    // every offered frame is visible to this call's outputs; how many are CONSUMED is decided once m is known
    const bool ending = s->ended || d->end_of_input;
    const double end_rel = (double)(s->total_in + n - s->origin_abs);
    const double P = s->spos;
    m = count_outputs(cap, [&](long long mm) {
        const double T = P + (double)mm * step;
        const long long i0 = (long long)std::floor(T);
        if (ending) return !(T + step > end_rel);
        return !(i0 + wc + 1 > have - 1);
    });
    // libsamplerate consumes only the input its outputs needed: when the output capacity ended the call, keep just
    // the frames the next output's window reaches and hand the rest back (bounded history for any ratio)
    long long used = n;
    if (m == cap) {
        const long long need = (long long)std::floor(P + (double)m * step) + wc + 2 - s->kept;
        used = need < 0 ? 0 : (need > n ? n : need);
    }
    const long long have_kept = s->kept + used;  // frames that stay in the handle after this call
    s->total_in += used;
    d->input_frames_used = (long)used;
    if (d->end_of_input && used == n) s->ended = true;
    L.v = (const float *)V2.p; L.have = have; L.origin = 0; L.pos = P; L.n_out = m;
    L.half_len = half_len; L.rq = rq; L.rho = rho; L.wc = wc;
    float *dout = d->data_out;
    if (!dev_ptrs) {
        rc = s->d_out.reserve(std::max<size_t>((size_t)m * fb, 16));
        if (rc) return rc;
        dout = (float *)s->d_out.p;
    }
    L.out = dout;
    rc = SDR_ERR_UNSUPPORTED;
    if (!s->exact && m >= SRC_FAST_MIN_OUT) rc = src_fast_run(s, L, st);
    if (rc == SDR_ERR_UNSUPPORTED) {
        if ((size_t)(wc + 6) * 64 * sizeof(double) <= ((size_t)64 << 20) && s->coef.reserve((size_t)(wc + 6) * 64 * sizeof(double)) == SDR_OK)
            L.coef = (double *)s->coef.p;
        rc = src_launch(L, st);
    }
    if (rc) return rc;
    if (!dev_ptrs && m > 0) SDR_CUDA_TRY(cudaMemcpyAsync(d->data_out, dout, (size_t)m * fb, cudaMemcpyDeviceToHost, st));
    d->output_frames_gen = (long)m;
    // rebase: keep wc+2 frames behind the next output position
    const double Pn = P + (double)m * step;
    long long drop = (long long)std::floor(Pn) - wc - 2;
    if (drop > have_kept) drop = have_kept;
    if (drop > 0) {
        const long long keep = have_kept - drop;
        rc = W2.reserve((size_t)std::max<long long>(keep, 1) * fb);
        if (rc) return rc;
        if (keep > 0)
            SDR_CUDA_TRY(cudaMemcpyAsync(W2.p, (char *)V2.p + (size_t)drop * fb, (size_t)keep * fb, cudaMemcpyDeviceToDevice, st));
        s->cur ^= 1;
        s->kept = keep;
        s->origin_abs += drop;
        s->spos = Pn - (double)drop;
    } else {
        s->kept = have_kept;
        s->spos = Pn;
    }
    if (!dev_ptrs) SDR_CUDA_TRY(cudaStreamSynchronize(st));
    return SDR_OK;
}

extern "C" int sdr_src_process(SDR_SRC_STATE *s, SDR_SRC_DATA *d) { return src_process_impl(s, d, false); }
extern "C" int sdr_src_process_dev(SDR_SRC_STATE *s, SDR_SRC_DATA *d) { return src_process_impl(s, d, true); }

// ============================================================================================
// timing helper
// ============================================================================================
struct sdr_timer {
    int dev;
    cudaStream_t st;
    cudaEvent_t a, b;
};
extern "C" sdr_timer_t *sdr_timer_create(int device, void *stream, int *err) {
    int dummy;
    if (!err) err = &dummy;
    if ((*err = check_device(device)) != SDR_OK) return nullptr;
    DeviceGuard g(device);
    sdr_timer *t = new sdr_timer;
    t->dev = device;
    t->st = (cudaStream_t)stream;
    if (cudaEventCreate(&t->a) != cudaSuccess || cudaEventCreate(&t->b) != cudaSuccess) {
        *err = SDR_ERR_CUDA_BASE;
        delete t;
        return nullptr;
    }
    return t;
}
extern "C" void sdr_timer_destroy(sdr_timer_t *t) {
    if (!t) return;
    DeviceGuard g(t->dev);
    cudaEventDestroy(t->a);
    cudaEventDestroy(t->b);
    delete t;
}
extern "C" int sdr_timer_begin(sdr_timer_t *t) {
    if (!t) return SDR_ERR_NULL_HANDLE;
    DeviceGuard g(t->dev);
    if (!g.ok) return g.status();
    return cuda_status(cudaEventRecord(t->a, t->st));
}
extern "C" int sdr_timer_end(sdr_timer_t *t, float *ms) {
    if (!t) return SDR_ERR_NULL_HANDLE;
    DeviceGuard g(t->dev);
    if (!g.ok) return g.status();
    SDR_CUDA_TRY(cudaEventRecord(t->b, t->st));
    SDR_CUDA_TRY(cudaEventSynchronize(t->b));
    return cuda_status(cudaEventElapsedTime(ms, t->a, t->b));
}

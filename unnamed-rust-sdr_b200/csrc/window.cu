// window.cu -- sdr_window_fft_*: the spectrum path of examples/live.rs:30-39
//     sig.window(duration).decimate(fps).map(|w| fft::fft(from_iter(rate, w.iter().cloned())))
// Window (src/signal/adapters/mod.rs:271-303) keeps the last cap = round(duration * rate) samples in a deque that
// starts as cap zeros and yields the deque after every input sample; Decimate (mod.rs:14-41) keeps every D-th of those
// (the one after input sample (k+1)*D - 1); fft::fft (src/fft.rs:3-28) transforms each kept window.  Here the kept
// windows of a block of input are gathered side by side in HBM (bytes unpacked on the way, rtltcp.rs:158-164) and go
// through one batched FFT of length cap (any length: Bluestein when not a power of two -- live.rs uses 1000).
// Carried across calls: the last cap - 1 input samples and the stream position, so blocks of any size may be fed.
#include <new>

#include "kernels.h"

using namespace sdr;

namespace {

// window w (stream-global index j0 + w) ends at input sample e = (j0 + w + 1) * D - 1 and holds samples e - N + 1 .. e;
// `buf` holds stream samples base .. base + have - 1 (history first); indices below 0 are the deque's initial zeros.
template <bool U8>
__global__ void window_gather_kernel(const void *__restrict__ buf, long long base, long long N, long long D,
                                     long long j0, float2 *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const long long w = blockIdx.y;
    const long long e = (j0 + w + 1) * D - 1;
    const long long idx = e - N + 1 + i;
    float2 v = make_float2(0.f, 0.f);
    if (idx >= 0) {
        if (U8) v = unpack_iq_u16(reinterpret_cast<const uint16_t *>(buf)[idx - base]);
        else v = reinterpret_cast<const float2 *>(buf)[idx - base];
    }
    out[w * N + i] = v;
}

}  // namespace

struct WindowHost {
    int dev = 0;
    size_t N = 0, D = 0;
    int fmt = SDR_FMT_C64;
    unsigned fft_flags = 0;
    long long total = 0;  // input samples seen
    long long kept = 0;   // history samples in d_buf (stream indices total - kept .. total - 1)
    long long emitted = 0;  // windows emitted so far
};

struct sdr_window_fft : WindowHost {
    StreamRef stream;
    Owned<sdr_fft_t, sdr_fft_destroy> plan;
    DevBuf d_buf[2], d_win, d_in, d_out;
    int cur = 0;

    int alloc(void *user_stream, const sdr_window_fft *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        sdr_fft_config_t fc;
        fc.n = N;
        fc.input_format = SDR_FMT_C64;  // the gather unpacks
        fc.flags = fft_flags;
        fc.device = dev;
        fc.stream = (void *)stream.s;
        plan.reset(sdr_fft_create(&fc, &rc));
        return plan ? SDR_OK : rc;
    }
};

extern "C" sdr_window_fft_t *sdr_window_fft_create(const sdr_window_fft_config_t *cfg, int *err) {
    if (!cfg || cfg->window == 0 || cfg->hop == 0 || cfg->window > ((size_t)1 << 26) ||
        (cfg->input_format != SDR_FMT_U8IQ && cfg->input_format != SDR_FMT_C64) || (cfg->flags & SDR_FFT_RFFT))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_window_fft>(err, cfg->device, cfg->stream, [&](sdr_window_fft &h) {
        h.N = cfg->window;
        h.D = cfg->hop;
        h.fmt = cfg->input_format;
        h.fft_flags = cfg->flags;
        return SDR_OK;
    });
}

extern "C" void sdr_window_fft_destroy(sdr_window_fft_t *h) { destroy_handle(h); }

extern "C" int sdr_window_fft_reset(sdr_window_fft_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    h->total = h->kept = h->emitted = 0;
    return SDR_OK;
}

extern "C" size_t sdr_window_fft_size(const sdr_window_fft_t *h) { return h ? h->N : 0; }

// windows that the next n_in samples complete: window j needs input sample (j + 1) * D - 1
extern "C" size_t sdr_window_fft_output_count(const sdr_window_fft_t *h, size_t n_in) {
    if (!h) return 0;
    const long long after = (h->total + (long long)n_in) / (long long)h->D;
    return (size_t)(after - h->emitted);
}

static int wf_run(sdr_window_fft *h, const void *in, size_t n_in, float *d_out, size_t out_cap, size_t *n_windows,
                  cudaMemcpyKind kin) {
    const size_t es = h->fmt == SDR_FMT_U8IQ ? 2 : 8;
    cudaStream_t st = h->stream.s;
    const long long N = (long long)h->N, D = (long long)h->D;
    const size_t nw = sdr_window_fft_output_count(h, n_in);
    if (nw > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    // stream samples base .. total + n_in - 1 side by side: history, then the new block
    const long long have = h->kept + (long long)n_in;
    DevBuf &A = h->d_buf[h->cur];
    DevBuf &B = h->d_buf[h->cur ^ 1];
    int rc = B.reserve((size_t)(have > 0 ? have : 1) * es + 16);
    if (rc) return rc;
    if (h->kept > 0) SDR_CUDA_TRY(cudaMemcpyAsync(B.p, A.p, (size_t)h->kept * es, cudaMemcpyDeviceToDevice, st));
    if (n_in > 0) SDR_CUDA_TRY(cudaMemcpyAsync((char *)B.p + (size_t)h->kept * es, in, n_in * es, kin, st));
    const long long base = h->total - h->kept;
    if (nw > 0) {
        rc = h->d_win.reserve(nw * (size_t)N * 8);
        if (rc) return rc;
        dim3 grid((unsigned)((N + 255) / 256), (unsigned)std::min<size_t>(nw, 65535));
        for (size_t w0 = 0; w0 < nw; w0 += 65535) {
            const size_t cnt = std::min<size_t>(65535, nw - w0);
            grid.y = (unsigned)cnt;
            float2 *dst = (float2 *)h->d_win.p + w0 * (size_t)N;
            if (h->fmt == SDR_FMT_U8IQ)
                window_gather_kernel<true><<<grid, 256, 0, st>>>(B.p, base, N, D, h->emitted + (long long)w0, dst);
            else
                window_gather_kernel<false><<<grid, 256, 0, st>>>(B.p, base, N, D, h->emitted + (long long)w0, dst);
            count_launch();
            rc = launch_status();
            if (rc) return rc;
        }
        rc = sdr_fft_exec_dev(h->plan.get(), h->d_win.p, nw, d_out);
        if (rc) return rc;
    }
    // keep the last N - 1 samples as history for the windows still to come
    h->total += (long long)n_in;
    h->emitted += (long long)nw;
    const long long keep = std::min<long long>(have, N - 1);
    if (keep > 0 && keep < have) {
        // move the tail to the front of the other buffer
        rc = A.reserve((size_t)keep * es + 16);
        if (rc) return rc;
        SDR_CUDA_TRY(cudaMemcpyAsync(A.p, (char *)B.p + (size_t)(have - keep) * es, (size_t)keep * es, cudaMemcpyDeviceToDevice, st));
        // A holds the history: cur stays
    } else {
        h->cur ^= 1;  // B holds everything and all of it is history
    }
    h->kept = keep;
    *n_windows = nw;
    return SDR_OK;
}

extern "C" int sdr_window_fft_process_dev(sdr_window_fft_t *h, const void *in, size_t n_in, float *out_c64,
                                          size_t out_cap, size_t *n_windows) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_windows || (n_in > 0 && !in) || !out_c64) return SDR_ERR_BAD_DATA_PTR;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    return wf_run(h, in, n_in, out_c64, out_cap, n_windows, cudaMemcpyDeviceToDevice);
}

extern "C" int sdr_window_fft_process(sdr_window_fft_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                                      size_t *n_windows) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_windows || (n_in > 0 && !in) || !out_c64) return SDR_ERR_BAD_DATA_PTR;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t nw = sdr_window_fft_output_count(h, n_in);
    if (nw > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    int rc = h->d_out.reserve(std::max<size_t>(nw * h->N * 8, 16));
    if (rc) return rc;
    rc = wf_run(h, in, n_in, (float *)h->d_out.p, out_cap, n_windows, cudaMemcpyHostToDevice);
    if (rc) return rc;
    if (nw > 0)
        SDR_CUDA_TRY(cudaMemcpyAsync(out_c64, h->d_out.p, nw * h->N * 8, cudaMemcpyDeviceToHost, h->stream.s));
    return cuda_status(cudaStreamSynchronize(h->stream.s));
}

// duc.cu -- K11, sdr_duc_*: digital up-converter bank, the transpose of sdr_ddc.  C channel streams, each zero-stuffed
// by I on sdr_pfs's grid (sample m at index (m+1) I - 1), filtered by its real taps h_k (Fir<f32, Complex<f32>>,
// src/filter/fir.rs:23-32), mixed UP by its 64-bit NCO and summed; F = first_sample is the absolute index of output 0:
//     u_k[n] = sum_{j<L} h_k[j] s_k[n - j],   x[n] = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64},  phi_k(N) = N Delta_k
// Computed form (filter, then rotate): write n = q I + c - 1, c = (n + 1) mod I; then
//     u_k[n] = sum_{i < I_c} h_k[c + i I] y_k[q - 1 - i],   I_c = ceil((L - c) / I)
// as one fmaf chain per component in ascending i (a tap of 0.0 is still multiplied, so NaNs propagate), and x[n] is
// accumulated over ascending k.  The rotation is one f64 sincospi of the exact integer phase per (tile, channel) times
// a per-channel f32 table built in f64 on the host.  Tiles of T outputs sit on the ABSOLUTE output grid, so an output's
// bits depend only on its frames and on F + n: blockings, clones and primed shards give the bits of one call.
// Carried across calls: the last H = ceil((L - 1) / I) frames of every channel and the stream position.
#include <algorithm>
#include <climits>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "nco.cuh"

using namespace sdr;

namespace {

constexpr size_t DUC_MAX_CH = 256;
constexpr size_t DUC_MAX_TAPS = (size_t)1 << 20;
constexpr int DUC_THREADS = 128;
constexpr int DUC_WIN = 8;                                   // outputs of one phase a thread keeps in registers
constexpr long long DUC_WIDE_TILE = 1024;                    // tile for I > 128 (one output per item)
constexpr size_t DUC_HOST_BYTES = (size_t)32 << 20;          // host-memory calls: chunk size of input and output

// Frame j (handle index) of channel k: 0 below lo (before the stream) and from end on, hist[k H + j - hist_lo] below
// y_lo (the carried frames), y[k stride + j - y_lo] from y_lo on (the caller's block, never copied).
struct DucSrc {
    const float2 *hist;
    const float2 *y;
    long long H, stride;
    long long lo, hist_lo, y_lo, end;
};

__device__ __forceinline__ float2 duc_load(const DucSrc &s, int k, long long j) {
    if (j < s.lo || j >= s.end) return make_float2(0.f, 0.f);
    if (j < s.y_lo) return __ldg(s.hist + k * s.H + (j - s.hist_lo));
    return __ldg(s.y + k * s.stride + (j - s.y_lo));
}

__device__ __forceinline__ long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// acc[w] = u_k of output phase c at frames qb + w (w < W): the sliding window holds y[qb - 1 - i + w] in slot
// (w - i) mod W, so every tap step loads one tap and one frame.  CHECK = false when every frame read lies in the block.
template <int W, bool CHECK>
__device__ __forceinline__ void duc_phase(const DucSrc &s, int k, const float *__restrict__ hk, long long I,
                                          long long c, int Ic, long long qb, float2 (&acc)[W]) {
    float2 win[W];
    const float2 *yk = s.y + k * s.stride - s.y_lo;  // frame j of the block at yk + j
#pragma unroll
    for (int w = 0; w < W; ++w) {
        acc[w] = make_float2(0.f, 0.f);
        const long long j = qb - 1 + w;
        win[w] = CHECK ? duc_load(s, k, j) : __ldg(yk + j);
    }
    const float *hp = hk + c;
    const float2 *yp = yk + (qb - 2);
    int i0 = 0;
    // whole groups of W taps without guards (the last one loads frame qb - 1 - Ic, which no tap uses)
    for (; i0 + W <= Ic; i0 += W) {
#pragma unroll
        for (int u = 0; u < W; ++u) {
            const int i = i0 + u;
            const float h = __ldg(hp);
            hp += I;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const float2 v = win[(w - u + W) % W];
                acc[w].x = __fmaf_rn(h, v.x, acc[w].x);
                acc[w].y = __fmaf_rn(h, v.y, acc[w].y);
            }
            win[(W - 1 - u) % W] = CHECK ? duc_load(s, k, qb - 2 - i) : __ldg(yp - i);
        }
    }
#pragma unroll
    for (int u = 0; u < W - 1; ++u) {
        const int i = i0 + u;
        if (i < Ic) {
            const float h = __ldg(hp);
            hp += I;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const float2 v = win[(w - u + W) % W];
                acc[w].x = __fmaf_rn(h, v.x, acc[w].x);
                acc[w].y = __fmaf_rn(h, v.y, acc[w].y);
            }
            if (i + 1 < Ic) win[(W - 1 - u) % W] = CHECK ? duc_load(s, k, qb - 2 - i) : __ldg(yp - i);
        }
    }
}

// One CTA per absolute tile of T outputs, tile tau of the call covering handle outputs [tau T - off, (tau+1) T - off).
// Item e (tile offset r = e mod I + (e / I) W I) owns the W outputs r + w I, all of phase c and frames qb + w; with
// W = 1 an item is one output.  base_s[k] = e^{+2 pi i (A_tile Delta_k) / 2^64}; output r of channel k is rotated by
// base_s[k] tab[k T + r].
template <int W>
__global__ void __launch_bounds__(DUC_THREADS) duc_kernel(DucSrc src, const float *__restrict__ taps, int tap_rows,
                                                          int L, const uint64_t *__restrict__ inc,
                                                          const float2 *__restrict__ tab, int C, long long I,
                                                          long long T, long long off, uint64_t a0, long long tau0,
                                                          long long n0, long long nt, float2 *__restrict__ out) {
    __shared__ float2 base_s[DUC_MAX_CH];
    const long long tau = tau0 + blockIdx.x;
    const long long nbase = tau * T - off;  // handle index of tile offset 0 (may be negative in the first tile)
    for (int k = threadIdx.x; k < C; k += blockDim.x) {
        float2 b = nco_rot((a0 + (uint64_t)tau * (uint64_t)T) * __ldg(inc + k));
        base_s[k] = make_float2(b.x, -b.y);
    }
    __syncthreads();
    const int items = (int)(T / W);
    for (int e = threadIdx.x; e < items; e += blockDim.x) {
        const long long r = e % I + (long long)(e / I) * W * I;
        const long long n1 = nbase + r + 1;
        const long long qb = floor_div(n1, I);
        const long long c = n1 - qb * I;
        const int Ic = c < L ? (int)((L - 1 - c) / I) + 1 : 0;
        // every frame this item reads (qb - 1 - Ic .. qb + W - 2) lies in the caller's block: no range checks
        const bool inside = qb - 1 - Ic >= src.y_lo && qb + W - 2 < src.end;
        float2 tot[W];
#pragma unroll
        for (int w = 0; w < W; ++w) tot[w] = make_float2(0.f, 0.f);
        for (int k = 0; k < C; ++k) {
            const float *hk = taps + (tap_rows == 1 ? 0 : (size_t)k * L);
            float2 acc[W];
            if (inside) duc_phase<W, false>(src, k, hk, I, c, Ic, qb, acc);
            else duc_phase<W, true>(src, k, hk, I, c, Ic, qb, acc);
            const float2 b = base_s[k];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const float2 rt = cmul(b, __ldg(tab + (size_t)k * T + r + w * I));
                tot[w].x = __fmaf_rn(-rt.y, acc[w].y, __fmaf_rn(rt.x, acc[w].x, tot[w].x));
                tot[w].y = __fmaf_rn(rt.y, acc[w].x, __fmaf_rn(rt.x, acc[w].y, tot[w].y));
            }
        }
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const long long n = nbase + r + w * I;
            if (r + w * I < T && n >= n0 && n < n0 + nt) out[n - n0] = tot[w];
        }
    }
}

// window and tile: W = DUC_WIN with T = I W floor(128 / I) (every phase has W outputs per item) for I <= 128, else
// one output per item and T = DUC_WIDE_TILE.  T <= 1024 either way.
void duc_geometry(size_t I, int *W, long long *T) {
    if (I <= (size_t)DUC_THREADS) {
        *W = DUC_WIN;
        *T = (long long)I * DUC_WIN * (DUC_THREADS / (long long)I);
    } else {
        *W = 1;
        *T = DUC_WIDE_TILE;
    }
}

}  // namespace

struct DucHost {
    int dev = 0;
    size_t L = 0, C = 0, I = 1, H = 0, n_sets = 1;
    uint64_t first = 0;
    int W = 1;
    long long T = 1;
    std::vector<float> taps;    // n_sets x L, as given
    std::vector<uint64_t> inc;
    long long total = 0;        // frames seen
};

struct sdr_duc : DucHost {
    StreamRef stream;
    DevBuf d_taps, d_inc, d_tab;
    DevBuf d_hist[2];           // C rows of the H frames before `total`
    int cur = 0;
    DevBuf d_in, d_out;

    // taps, increments, rotation tables (f64 on the host, rounded to f32 once) and history of a handle whose fields are set
    int alloc(void *user_stream, const sdr_duc *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        cudaStream_t st = stream.s;
        duc_geometry(I, &W, &T);
        std::vector<float2> tab((size_t)C * T);
        for (size_t k = 0; k < C; ++k)
            for (long long r = 0; r < T; ++r) {
                const double t = NCO_2PI * nco_turns((uint64_t)r * inc[k]);
                tab[k * T + r] = make_float2((float)std::cos(t), (float)std::sin(t));
            }
        if ((rc = d_taps.upload(taps.data(), taps.size() * sizeof(float), st))) return rc;
        if ((rc = d_inc.upload(inc.data(), C * sizeof(uint64_t), st))) return rc;
        if ((rc = d_tab.upload(tab.data(), tab.size() * sizeof(float2), st))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(H, 1) * C * 8))) return rc;
        return cuda_status(cudaStreamSynchronize(st));
    }
    int copy_device(const sdr_duc &src) {
        if (H == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, H * C * 8, cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_duc_t *sdr_duc_create(const sdr_duc_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || !cfg->phase_inc || cfg->n_taps == 0 || cfg->n_taps > DUC_MAX_TAPS ||
        cfg->n_channels == 0 || cfg->n_channels > DUC_MAX_CH ||
        (cfg->n_tap_sets != 1 && cfg->n_tap_sets != cfg->n_channels) || cfg->interpolation == 0 ||
        cfg->interpolation > ((size_t)1 << 40) || cfg->flags != 0)
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_duc>(err, cfg->device, cfg->stream, [&](sdr_duc &h) {
        h.L = cfg->n_taps;
        h.C = cfg->n_channels;
        h.I = cfg->interpolation;
        h.H = (h.L - 1 + h.I - 1) / h.I;
        h.n_sets = cfg->n_tap_sets;
        h.first = cfg->first_sample;
        h.taps.assign(cfg->taps, cfg->taps + h.L * h.n_sets);
        h.inc.assign(cfg->phase_inc, cfg->phase_inc + h.C);
        return SDR_OK;
    });
}

extern "C" void sdr_duc_destroy(sdr_duc_t *h) { destroy_handle(h); }

extern "C" int sdr_duc_reset(sdr_duc_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // frames below 0 read as zero, so the stale history is never used
    h->total = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_duc_t *sdr_duc_clone(const sdr_duc_t *src, int *err) { return clone_handle<DucHost>(src, err); }

extern "C" size_t sdr_duc_output_count(const sdr_duc_t *h, size_t n_frames) {
    if (!h) return 0;
    return n_frames * h->I;
}

// in: C device rows of nf frames, row stride in_stride; out: nf * I samples
static int duc_run(sdr_duc *h, const float2 *in, size_t nf, size_t in_stride, float2 *out) {
    cudaStream_t st = h->stream.s;
    const long long I = (long long)h->I, T = h->T, H = (long long)h->H;
    DucSrc s;
    s.hist = (const float2 *)h->d_hist[h->cur].p;
    s.y = in;
    s.H = H;
    s.stride = (long long)in_stride;
    s.y_lo = h->total;
    s.hist_lo = h->total - H;
    s.lo = std::max(0LL, s.hist_lo);
    s.end = h->total + (long long)nf;
    const long long n0 = h->total * I, nt = (long long)nf * I;
    const long long off = (long long)(h->first % (uint64_t)T);
    const uint64_t a0 = h->first - (uint64_t)off;
    const long long tau0 = (n0 + off) / T, tau1 = (n0 + nt - 1 + off) / T;
    for (long long t0 = tau0; t0 <= tau1; t0 += 1LL << 30) {
        const unsigned grid = (unsigned)std::min(tau1 - t0 + 1, 1LL << 30);
        if (h->W == DUC_WIN)
            duc_kernel<DUC_WIN><<<grid, DUC_THREADS, 0, st>>>(s, (const float *)h->d_taps.p, (int)h->n_sets, (int)h->L,
                                                            (const uint64_t *)h->d_inc.p, (const float2 *)h->d_tab.p,
                                                            (int)h->C, I, T, off, a0, t0, n0, nt, out);
        else
            duc_kernel<1><<<grid, DUC_THREADS, 0, st>>>(s, (const float *)h->d_taps.p, (int)h->n_sets, (int)h->L,
                                                      (const uint64_t *)h->d_inc.p, (const float2 *)h->d_tab.p,
                                                      (int)h->C, I, T, off, a0, t0, n0, nt, out);
        count_launch();
        int rc = launch_status();
        if (rc) return rc;
    }
    // history = the last H frames of (history, block), per channel
    if (H > 0) {
        const size_t from_y = std::min(nf, (size_t)H), from_old = (size_t)H - from_y;
        char *dst = (char *)h->d_hist[h->cur ^ 1].p;
        if (from_old > 0)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(dst, H * 8, (const char *)h->d_hist[h->cur].p + from_y * 8, H * 8,
                                           from_old * 8, h->C, cudaMemcpyDeviceToDevice, st));
        SDR_CUDA_TRY(cudaMemcpy2DAsync(dst + from_old * 8, H * 8, in + (nf - from_y), in_stride * 8, from_y * 8, h->C,
                                       cudaMemcpyDeviceToDevice, st));
        h->cur ^= 1;
    }
    h->total += (long long)nf;
    return SDR_OK;
}

static int duc_check(const sdr_duc *h, const float *in, size_t n_frames, size_t in_stride, const float *out,
                     size_t out_cap, size_t *n_out) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    *n_out = 0;
    if (n_frames == 0) return SDR_OK;
    if (!in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < n_frames) return SDR_ERR_INVALID_ARG;
    // handle output indices stay within int64: (total + n_frames) I
    const unsigned long long lim = (unsigned long long)LLONG_MAX / h->I;
    if (n_frames > lim || (unsigned long long)h->total + n_frames > lim) return SDR_ERR_INVALID_ARG;
    if (sdr_duc_output_count(h, n_frames) > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (!out) return SDR_ERR_BAD_DATA_PTR;
    return SDR_OK;
}

extern "C" int sdr_duc_process_dev(sdr_duc_t *h, const float *in_c64, size_t n_frames, size_t in_stride,
                                   float *out_c64, size_t out_cap, size_t *n_out) {
    int rc = duc_check(h, in_c64, n_frames, in_stride, out_c64, out_cap, n_out);
    if (rc || n_frames == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = duc_run(h, (const float2 *)in_c64, n_frames, h->C > 1 ? in_stride : n_frames, (float2 *)out_c64);
    if (rc) return rc;
    *n_out = n_frames * h->I;
    return SDR_OK;
}

extern "C" int sdr_duc_process(sdr_duc_t *h, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                               size_t out_cap, size_t *n_out) {
    int rc = duc_check(h, in_c64, n_frames, in_stride, out_c64, out_cap, n_out);
    if (rc || n_frames == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C, I = h->I;
    const size_t stride = C > 1 ? in_stride : n_frames;
    cudaStream_t st = h->stream.s;
    // chunks of about DUC_HOST_BYTES of input and of output: H2D, compute, D2H in stream order
    size_t chunk = std::max<size_t>(1, std::min(DUC_HOST_BYTES / (C * 8), DUC_HOST_BYTES / (I * 8)));
    chunk = std::min(chunk, n_frames);
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_out.reserve(chunk * I * 8);
    if (rc) return rc;
    for (size_t done = 0; done < n_frames;) {
        const size_t cnt = std::min(chunk, n_frames - done);
        SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, cnt * 8, in_c64 + done * 2, stride * 8, cnt * 8, C,
                                       cudaMemcpyHostToDevice, st));
        rc = duc_run(h, (const float2 *)h->d_in.p, cnt, cnt, (float2 *)h->d_out.p);
        if (rc) return rc;
        SDR_CUDA_TRY(cudaMemcpyAsync(out_c64 + done * I * 2, h->d_out.p, cnt * I * 8, cudaMemcpyDeviceToHost, st));
        done += cnt;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_out = n_frames * I;
    return SDR_OK;
}

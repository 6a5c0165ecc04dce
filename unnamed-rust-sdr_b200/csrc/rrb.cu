// rrb.cu -- K13, sdr_rrb_*: rational resampler bank.  C independent c64 channel streams, channel k resampled by its own
// I_k / D_k with real taps h_k: zero-stuffed on sdr_pfs's grid, filtered by Fir<f32, Complex<f32>> (src/filter/fir.rs:
// 23-32) and decimated by signal::Decimate (adapters/mod.rs:30-37); m counts the handle's frames, frames before 0 are 0:
//     s_k[(m+1) I_k - 1] = y_k[m],   u_k[n] = sum_{j<L} h_k[j] s_k[n - j],   z_k[r] = u_k[(r+1) D_k - 1]
// Computed form: t = (r+1) D - 1, q = (t+1) div I, c = (t+1) mod I;
//     z_k[r] = sum_{i < I_c} h_k[c + i I] y_k[q - 1 - i],   I_c = ceil((L - c) / I)
// as one fmaf chain per component in ascending i (a tap of 0.0 is still multiplied, so NaNs propagate; taps past L never
// are).  With g = gcd(I, D) the chain of (g I', g D', h) has the same terms in the same order as that of (I', D', h[g j]),
// so create reduces every channel and builds one phase-major table per distinct (tap set, I', g): row c holds
// h[g (c + i I')], i < I_c, with no padding.  An output is one fixed chain, so its bits do not depend on blocking.
// Counts: after n frames a channel has released floor(n I / D) outputs (128-bit on the host).
// Carried across calls: the last H_k = ceil(L'_k / I'_k) frames of every channel and its frame count.
#include <algorithm>
#include <climits>
#include <map>
#include <new>
#include <numeric>
#include <tuple>
#include <vector>

#include "bank.cuh"
#include "kernels.h"

using namespace sdr;

namespace {

constexpr size_t RRB_MAX_CH = 65536;
constexpr size_t RRB_MAX_TAPS = (size_t)1 << 20;
constexpr size_t RRB_MAX_TAP_FLOATS = (size_t)1 << 26;
constexpr size_t RRB_MAX_I = (size_t)1 << 16;
constexpr size_t RRB_MAX_D = (size_t)1 << 24;
constexpr unsigned long long RRB_MAX_POS = 1ull << 62;  // frame counts and n I per call stay below this
constexpr int RRB_THREADS = 128;
constexpr int RRB_R = 4;                                 // outputs of one phase per thread (windows D' frames apart)
constexpr size_t RRB_HOST_BYTES = (size_t)32 << 20;      // host-memory calls: chunk size of input

struct RrbChan {   // per channel, fixed at create (reduced ratio)
    double rI;     // 1 / I'
    long long D;   // D'
    long long tab; // offset of the channel's phase-major table in the tap buffer
    long long hist;// offset of the channel's H carried frames in a history buffer
    int I, L, H;   // I', L' = ceil(L / g), H = ceil(L' / I')
    int pad;
};

struct RrbCall {    // per channel and call; frame indices are relative to the call's first frame
    long long qb;   // q of the call's output 0 (output e has q = qb + (c0 + e D') div I' and phase (c0 + e D') mod I')
    long long c0;
    long long cnt;  // outputs of the call
    long long n;    // frames of the call
    long long lo;   // frames below lo lie before the stream and read as 0
};

// frame j of a channel: hist[j] for j < 0 (hist points one past the carried frames), y[j] for 0 <= j < n, else 0
__device__ __forceinline__ float2 rrb_load(const float2 *hist, const float2 *y, long long j, long long lo, long long n) {
    if (j < lo || j >= n) return make_float2(0.f, 0.f);
    if (j < 0) return __ldg(hist + j);
    return __ldg(y + j);
}

// floor(x / d) and x mod d for 0 <= x < 2^52 and d <= 2^16 (rd = 1 / d): the f64 quotient is off by at most one, which
// one step corrects.  A 64-bit integer division would be a subroutine call.
__device__ __forceinline__ long long rrb_divmod(long long x, long long d, double rd, long long *m) {
    long long q = (long long)((double)x * rd);
    long long r = x - q * d;
    if (r < 0) { --q; r += d; }
    else if (r >= d) { ++q; r -= d; }
    *m = r;
    return q;
}

// acc[w] = the chain of the output whose q is q0 + w D (all R outputs share the phase, hence the taps hc[0..Ic)).
// CHECK = false when every frame read lies in the caller's row.
template <bool CHECK>
__device__ __forceinline__ void rrb_chain(const float *__restrict__ hc, int Ic, const float2 *hist, const float2 *y,
                                          long long q0, long long D, long long lo, long long n, float2 (&acc)[RRB_R]) {
#pragma unroll
    for (int w = 0; w < RRB_R; ++w) acc[w] = make_float2(0.f, 0.f);
    const float2 *yp = y + (q0 - 1);
    for (int i = 0; i < Ic; ++i) {
        const float h = __ldg(hc + i);
#pragma unroll
        for (int w = 0; w < RRB_R; ++w) {
            const float2 v = CHECK ? rrb_load(hist, y, q0 - 1 - i + w * D, lo, n) : __ldg(yp - i + w * D);
            acc[w].x = __fmaf_rn(h, v.x, acc[w].x);
            acc[w].y = __fmaf_rn(h, v.y, acc[w].y);
        }
    }
}

// One CTA per tile of RRB_THREADS items over the flattened (channel, item) space: channel k owns tiles
// [tile0[k], tile0[k+1]).  Item u of a channel is phase class p = u mod I' of output group u div I' (groups of R I'
// outputs): the outputs e0 + w I', w < R, e0 = (u div I') R I' + p, which share one phase and whose frames are D' apart.
// Consecutive lanes take consecutive p, so with I' > 1 they read different tap rows.
__global__ void __launch_bounds__(RRB_THREADS) rrb_kernel(const float *__restrict__ taps,
                                                          const RrbChan *__restrict__ chans,
                                                          const RrbCall *__restrict__ calls,
                                                          const long long *__restrict__ tile0, int C, long long tiles,
                                                          const float2 *__restrict__ hist,
                                                          const float2 *__restrict__ in, long long in_stride,
                                                          float2 *__restrict__ out, long long out_stride) {
    __shared__ int k_s;
    for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
        if (threadIdx.x == 0) k_s = bank_tile_channel(tile0, C, t);
        __syncthreads();
        const int k = k_s;
        __syncthreads();
        const RrbChan ch = chans[k];
        const RrbCall cl = calls[k];
        const long long I = ch.I;
        const long long u = (t - __ldg(tile0 + k)) * RRB_THREADS + threadIdx.x;
        long long p, cm;
        const long long grp = rrb_divmod(u, I, ch.rI, &p);
        const long long e0 = grp * I * RRB_R + p;
        if (e0 >= cl.cnt) continue;
        // (c0 + e0 D') div I' = grp R D' + (c0 + p D') div I', and c0 + p D' < 2^41
        const long long q0 = cl.qb + grp * RRB_R * ch.D + rrb_divmod(cl.c0 + p * ch.D, I, ch.rI, &cm);
        const int c = (int)cm;
        const int Ic = c < ch.L ? (ch.L - 1 - c) / ch.I + 1 : 0;
        // row c of the phase-major table starts at sum_{c' < c} I_c' = c floor(L' / I') + min(c, L' mod I')
        const float *hc = taps + ch.tab + (long long)c * (ch.L / ch.I) + min(c, ch.L % ch.I);
        const float2 *y = in + k * in_stride;
        const float2 *hk = hist + ch.hist + ch.H;
        const bool full = e0 + (RRB_R - 1) * I < cl.cnt;
        float2 acc[RRB_R];
        if (full && q0 - Ic >= 0 && q0 + (RRB_R - 1) * ch.D - 1 < cl.n)
            rrb_chain<false>(hc, Ic, hk, y, q0, ch.D, cl.lo, cl.n, acc);
        else
            rrb_chain<true>(hc, Ic, hk, y, q0, ch.D, cl.lo, cl.n, acc);
        float2 *o = out + k * out_stride + e0;
#pragma unroll
        for (int w = 0; w < RRB_R; ++w)
            if (e0 + w * I < cl.cnt) o[w * I] = acc[w];
    }
}

// history: the last H frames of (carried frames, the call's row), per channel; one CTA per channel
__global__ void __launch_bounds__(RRB_THREADS) rrb_carry_kernel(const RrbChan *__restrict__ chans,
                                                                const RrbCall *__restrict__ calls,
                                                                const float2 *__restrict__ hist_old,
                                                                const float2 *__restrict__ in, long long in_stride,
                                                                float2 *__restrict__ hist_new) {
    const int k = blockIdx.x;
    const RrbChan ch = chans[k];
    bank_carry(hist_old, in + k * in_stride, calls[k].n, ch.H, ch.hist, hist_new);
}

unsigned long long gcd_ull(unsigned long long a, unsigned long long b) {
    while (b) {
        const unsigned long long t = a % b;
        a = b;
        b = t;
    }
    return a;
}

}  // namespace

struct RrbHost {
    int dev = 0;
    size_t C = 0;
    std::vector<RrbChan> chans;             // reduced ratios, table and history offsets
    std::vector<unsigned long long> total;  // frames seen, per channel
    std::vector<float> tab;                 // every phase-major table
    size_t hist_len = 0;                    // sum of H_k
};

struct sdr_rrb : RrbHost {
    StreamRef stream;
    DevBuf d_tab, d_chans, d_call, d_hist[2];
    int cur = 0;
    std::vector<char> call_host;            // tile0 (C + 1) then C RrbCall, uploaded once per call
    DevBuf d_in, d_out;

    int alloc(void *user_stream, const sdr_rrb *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_tab.upload(tab.data(), tab.size() * sizeof(float), stream.s))) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(RrbChan), stream.s))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(hist_len, 1) * 8))) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_rrb &src) {
        if (hist_len == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, hist_len * 8, cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_rrb_t *sdr_rrb_create(const sdr_rrb_config_t *cfg, int *err) {
    bool ok = cfg && cfg->taps && cfg->interpolation && cfg->decimation && cfg->n_taps >= 1 &&
              cfg->n_taps <= RRB_MAX_TAPS && cfg->n_channels >= 1 && cfg->n_channels <= RRB_MAX_CH &&
              (cfg->n_tap_sets == 1 || cfg->n_tap_sets == cfg->n_channels) &&
              cfg->n_tap_sets * cfg->n_taps <= RRB_MAX_TAP_FLOATS;
    for (size_t k = 0; ok && k < cfg->n_channels; ++k)
        ok = cfg->interpolation[k] >= 1 && cfg->interpolation[k] <= RRB_MAX_I && cfg->decimation[k] >= 1 &&
             cfg->decimation[k] <= RRB_MAX_D;
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_rrb>(err, cfg->device, cfg->stream, [&](sdr_rrb &h) {
        h.C = cfg->n_channels;
        h.chans.resize(h.C);
        h.total.assign(h.C, 0);
        const size_t L = cfg->n_taps;
        // one phase-major table per distinct (tap set, I', g)
        std::map<std::tuple<size_t, size_t, size_t>, long long> tables;
        for (size_t k = 0; k < h.C; ++k) {
            const size_t I = cfg->interpolation[k], D = cfg->decimation[k], g = (size_t)gcd_ull(I, D);
            const size_t Ir = I / g, Lr = (L + g - 1) / g, set = cfg->n_tap_sets == 1 ? 0 : k;
            RrbChan &ch = h.chans[k];
            ch.I = (int)Ir;
            ch.rI = 1.0 / (double)Ir;
            ch.D = (long long)(D / g);
            ch.L = (int)Lr;
            ch.H = (int)((Lr + Ir - 1) / Ir);
            ch.pad = 0;
            ch.hist = (long long)h.hist_len;
            h.hist_len += (size_t)ch.H;
            const auto key = std::make_tuple(set, Ir, g);
            auto it = tables.find(key);
            if (it == tables.end()) {
                const float *src = cfg->taps + set * L;
                const long long at = (long long)h.tab.size();
                for (size_t c = 0; c < Ir; ++c)
                    for (size_t j = c; j < Lr; j += Ir) h.tab.push_back(src[g * j]);
                it = tables.emplace(key, at).first;
            }
            ch.tab = it->second;
        }
        return SDR_OK;
    });
}

extern "C" void sdr_rrb_destroy(sdr_rrb_t *h) { destroy_handle(h); }

extern "C" int sdr_rrb_reset(sdr_rrb_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // frames before the stream read as zero, so the stale history is never used
    std::fill(h->total.begin(), h->total.end(), 0ull);
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_rrb_t *sdr_rrb_clone(const sdr_rrb_t *src, int *err) { return clone_handle<RrbHost>(src, err); }

static unsigned long long rrb_released(const RrbChan &ch, unsigned long long frames) {
    return (unsigned long long)((unsigned __int128)frames * (unsigned)ch.I / (unsigned long long)ch.D);
}

extern "C" int sdr_rrb_output_count(const sdr_rrb_t *h, const size_t *n_in, size_t *counts) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !counts) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) {
        if (n_in[k] > RRB_MAX_POS - h->total[k]) return SDR_ERR_INVALID_ARG;
        counts[k] = (size_t)(rrb_released(h->chans[k], h->total[k] + n_in[k]) - rrb_released(h->chans[k], h->total[k]));
    }
    return SDR_OK;
}

// in: C device rows (row stride in_stride), row k of n_in[k] frames; out: C rows of out_stride, cnt[k] outputs each
static int rrb_run(sdr_rrb *h, const float2 *in, const size_t *n_in, size_t in_stride, const size_t *cnt, float2 *out,
                   size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    h->call_host.resize((C + 1) * sizeof(long long) + C * sizeof(RrbCall));
    long long *tile0 = (long long *)h->call_host.data();
    RrbCall *calls = (RrbCall *)(tile0 + C + 1);
    long long tiles = 0;
    bool any = false;
    for (size_t k = 0; k < C; ++k) {
        const RrbChan &ch = h->chans[k];
        const unsigned long long T = h->total[k];
        // (R0 + 1) D' = Q0 I' + c0 for the call's first output R0 = floor(T I' / D')
        const unsigned __int128 a = ((unsigned __int128)rrb_released(ch, T) + 1) * (unsigned long long)ch.D;
        const unsigned long long Q0 = (unsigned long long)(a / (unsigned)ch.I);
        RrbCall &cl = calls[k];
        cl.qb = (long long)(Q0 - T);  // 0 <= Q0 - T <= D' / I'
        cl.c0 = (long long)(a - (unsigned __int128)Q0 * (unsigned)ch.I);
        cl.cnt = (long long)cnt[k];
        cl.n = (long long)n_in[k];
        cl.lo = -(long long)std::min<unsigned long long>((unsigned long long)ch.H, T);
        any = any || n_in[k] > 0;
        // items: I' per full group of R I' outputs, then min(I', what is left)
        const long long G = (long long)ch.I * RRB_R, full = cl.cnt / G;
        const long long items = full * ch.I + std::min<long long>(ch.I, cl.cnt - full * G);
        tile0[k] = tiles;
        tiles += (items + RRB_THREADS - 1) / RRB_THREADS;
    }
    tile0[C] = tiles;
    if (!any) return SDR_OK;
    int rc = h->d_call.reserve(h->call_host.size());
    if (rc) return rc;
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_call.p, h->call_host.data(), h->call_host.size(), cudaMemcpyHostToDevice, st));
    const long long *d_tile0 = (const long long *)h->d_call.p;
    const RrbCall *d_calls = (const RrbCall *)(d_tile0 + C + 1);
    const long long stride = C > 1 ? (long long)in_stride : 0;
    if (tiles > 0) {
        const unsigned grid = (unsigned)std::min<long long>(tiles, 1LL << 30);
        rrb_kernel<<<grid, RRB_THREADS, 0, st>>>((const float *)h->d_tab.p, (const RrbChan *)h->d_chans.p, d_calls,
                                                 d_tile0, (int)C, tiles, (const float2 *)h->d_hist[h->cur].p, in,
                                                 stride, out, (long long)out_stride);
        count_launch();
        if ((rc = launch_status())) return rc;
    }
    if (h->hist_len > 0) {
        rrb_carry_kernel<<<(unsigned)C, RRB_THREADS, 0, st>>>((const RrbChan *)h->d_chans.p, d_calls,
                                                              (const float2 *)h->d_hist[h->cur].p, in, stride,
                                                              (float2 *)h->d_hist[h->cur ^ 1].p);
        count_launch();
        if ((rc = launch_status())) return rc;
        h->cur ^= 1;
    }
    for (size_t k = 0; k < C; ++k) h->total[k] += n_in[k];
    return SDR_OK;
}

static int rrb_check(const sdr_rrb *h, const float *in, const size_t *n_in, size_t in_stride, const float *out,
                     size_t out_cap, size_t out_stride, size_t *n_out, std::vector<size_t> &cnt, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out || !n_in) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = 0;
    *longest = *std::max_element(n_in, n_in + h->C);
    if (*longest > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < *longest) return SDR_ERR_INVALID_ARG;
    for (size_t k = 0; k < h->C; ++k)
        if (n_in[k] > RRB_MAX_POS / (unsigned)h->chans[k].I) return SDR_ERR_INVALID_ARG;
    cnt.resize(h->C);
    int rc = sdr_rrb_output_count(h, n_in, cnt.data());
    if (rc) return rc;
    const size_t most = *std::max_element(cnt.begin(), cnt.end());
    if (most > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (most > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (most > 0 && h->C > 1 && out_stride < most) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_rrb_process_dev(sdr_rrb_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                   float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    size_t longest = 0;
    int rc = rrb_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, cnt, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = rrb_run(h, (const float2 *)in_c64, n_in, in_stride, cnt.data(), (float2 *)out_c64, out_stride);
    if (rc) return rc;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = cnt[k];
    return SDR_OK;
}

extern "C" int sdr_rrb_process(sdr_rrb_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                               float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    size_t longest = 0;
    int rc = rrb_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, cnt, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t stride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : out_cap;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` frames per channel: H2D, compute, D2H in stream order
    const size_t chunk = std::min(longest, std::max<size_t>(1, RRB_HOST_BYTES / (C * 8)));
    const bool equal_in = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    std::vector<size_t> take(C), part(C), done(C, 0);
    size_t fcap = 0;
    for (size_t k = 0; k < C; ++k) {
        const unsigned long long lim = (unsigned long long)chunk * (unsigned)h->chans[k].I / h->chans[k].D + 1;
        fcap = std::max<size_t>(fcap, std::min<unsigned long long>(lim, cnt[k]));
    }
    fcap = std::max<size_t>(fcap, 1);
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_out.reserve(fcap * C * 8);
    if (rc) return rc;
    for (size_t pos = 0; pos < longest; pos += chunk) {
        for (size_t k = 0; k < C; ++k) take[k] = n_in[k] > pos ? std::min(chunk, n_in[k] - pos) : 0;
        if (equal_in)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, chunk * 8, in_c64 + 2 * pos, stride * 8, take[0] * 8, C,
                                           cudaMemcpyHostToDevice, st));
        else
            for (size_t k = 0; k < C; ++k)
                if (take[k])
                    SDR_CUDA_TRY(cudaMemcpyAsync((float2 *)h->d_in.p + k * chunk, in_c64 + 2 * (k * stride + pos),
                                                 take[k] * 8, cudaMemcpyHostToDevice, st));
        if ((rc = sdr_rrb_output_count(h, take.data(), part.data()))) return rc;
        rc = rrb_run(h, (const float2 *)h->d_in.p, take.data(), chunk, part.data(), (float2 *)h->d_out.p, fcap);
        if (rc) return rc;
        const bool equal_out = std::all_of(part.begin(), part.end(), [&](size_t p) { return p == part[0]; }) &&
                               std::all_of(done.begin(), done.end(), [&](size_t d) { return d == done[0]; });
        if (equal_out && part[0] > 0)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(out_c64 + 2 * done[0], ostride * 8, h->d_out.p, fcap * 8, part[0] * 8, C,
                                           cudaMemcpyDeviceToHost, st));
        else if (!equal_out)
            for (size_t k = 0; k < C; ++k)
                if (part[k])
                    SDR_CUDA_TRY(cudaMemcpyAsync(out_c64 + 2 * (k * ostride + done[k]), (float2 *)h->d_out.p + k * fcap,
                                                 part[k] * 8, cudaMemcpyDeviceToHost, st));
        for (size_t k = 0; k < C; ++k) done[k] += part[k];
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    for (size_t k = 0; k < C; ++k) n_out[k] = cnt[k];
    return SDR_OK;
}

// arb.cu -- K14, sdr_arb_*: arbitrary-ratio resampler bank.  C independent c64 channel streams; channel k has real taps
// h_k of length L designed at P = 2^p times the input rate, a step sigma_k and a first position tau_k(0), all positions
// exact in units of 2^-64 frames (m counts the handle's frames of the channel, frames before the stream are 0):
//     tau_k(r) = tau_k(0) + r sigma_k
//     H_k(t) = (1 - a) h_k[j] + a h_k[j+1],  j = floor(t P), a = t P - j,  0 <= j < L (h_k[L] = 0); 0 otherwise
//     z_k[r] = sum_{0 <= m <= floor(tau_k(r))} H_k(tau_k(r) - m) y_k[m]
// Computed form: n0 = floor(tau), f = its 64-bit fraction, ip = f >> (64 - p) (0 when P = 1),
// a = ((f << p) >> 40) 2^-24 (exact in f32), d_k[j] = f32(h_k[j+1] - h_k[j]) in f64 at create, and
//     c_i = fmaf(a, d_k[i P + ip], h_k[i P + ip]),   acc = fmaf(c_i, y_k[n0 - i], acc)   for i = 0, 1, ... while iP+ip < L
// one chain per component: frames before the stream are 0 and still multiplied, taps past L never are.  An output is
// one fixed chain, so its bits depend only on its inputs and its absolute position, not on blocking.
// Counts: after n frames a channel has released #{r : tau(r) < n} outputs (128-bit on the host).  set_steps starts a
// new segment at the next unreleased output: tau(R + e) = tau_old(R) + e sigma_new.
// Carried across calls: the last H_k = ceil(L / P) frames of every channel, its frame count and its time-base segment.
#include <algorithm>
#include <cmath>
#include <map>
#include <new>
#include <vector>

#include "arb_core.cuh"
#include "bank.cuh"
#include "kernels.h"

using namespace sdr;

namespace {

typedef unsigned __int128 u128;

constexpr size_t ARB_MAX_CH = 65536;
constexpr size_t ARB_MAX_TAPS = (size_t)1 << 20;
constexpr size_t ARB_MAX_TAP_FLOATS = (size_t)1 << 26;
constexpr size_t ARB_MAX_P = (size_t)1 << 16;
constexpr u128 ARB_MIN_STEP = (u128)1 << 48;            // 2^-16 frames
constexpr u128 ARB_MAX_STEP = (u128)1 << 88;            // 2^24 frames
constexpr unsigned long long ARB_MAX_POS = 1ull << 62;  // whole parts, frame totals and per-call counts stay below
constexpr int ARB_THREADS = 128;
constexpr size_t ARB_HOST_BYTES = (size_t)32 << 20;     // host-memory calls: chunk size of input

struct ArbChan {        // per channel, fixed at create
    long long tab;      // offset (float2 entries) of the channel's (h, d) table
    long long hist;     // offset of the channel's H carried frames in a history buffer
    int L, H, p, pad;   // taps, ceil(L / P), log2 P
};

struct ArbCall {                  // per channel and call; frames are relative to the call's first frame
    unsigned long long aw, af;    // tau of the call's output 0 minus the frames before the call (whole, fraction)
    unsigned long long sw, sf;    // the step
    long long cnt;                // outputs of the call
    long long n;                  // frames of the call
    long long lo;                 // frames below lo lie before the stream and read as 0
    long long pad;
};

// One CTA per tile of ARB_THREADS consecutive outputs over the flattened (channel, output) space: channel k owns tiles
// [tile0[k], tile0[k+1]).  Lane e of a tile takes output e, so a warp's frame loads span about 32 sigma frames.
__global__ void __launch_bounds__(ARB_THREADS) arb_kernel(const float2 *__restrict__ tab,
                                                          const ArbChan *__restrict__ chans,
                                                          const ArbCall *__restrict__ calls,
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
        const ArbCall cl = calls[k];
        const unsigned long long e = (unsigned long long)((t - __ldg(tile0 + k)) * ARB_THREADS + threadIdx.x);
        if ((long long)e >= cl.cnt) continue;
        const ArbChan ch = chans[k];
        // tau = anchor + e sigma in 64.64 integers (the whole part stays below 2^62)
        const unsigned long long lo = e * cl.sf;
        const unsigned long long f = cl.af + lo;
        const long long n0 = (long long)(cl.aw + e * cl.sw + __umul64hi(e, cl.sf) + (f < lo ? 1ull : 0ull));
        const int ip = ch.p ? (int)(f >> (64 - ch.p)) : 0;
        const float a = (float)((f << ch.p) >> 40) * 0x1p-24f;
        const int P = 1 << ch.p;
        const int T = ip < ch.L ? ((ch.L - ip + P - 1) >> ch.p) : 0;
        const float2 *tb = tab + ch.tab + ip;
        const float2 *y = in + k * in_stride;
        const float2 *hk = hist + ch.hist + ch.H;
        const float2 z = n0 - ch.H + 1 >= 0 ? arb_chain<false>(tb, T, P, a, hk, y, n0, cl.lo)
                                            : arb_chain<true>(tb, T, P, a, hk, y, n0, cl.lo);
        out[k * out_stride + (long long)e] = z;
    }
}

// history: the last H frames of (carried frames, the call's row), per channel; one CTA per channel
__global__ void __launch_bounds__(ARB_THREADS) arb_carry_kernel(const ArbChan *__restrict__ chans,
                                                                const ArbCall *__restrict__ calls,
                                                                const float2 *__restrict__ hist_old,
                                                                const float2 *__restrict__ in, long long in_stride,
                                                                float2 *__restrict__ hist_new) {
    const int k = blockIdx.x;
    const ArbChan ch = chans[k];
    bank_carry(hist_old, in + k * in_stride, calls[k].n, ch.H, ch.hist, hist_new);
}

u128 to_u128(const sdr_arb_time_t &t) { return ((u128)t.whole << 64) | t.frac; }

bool step_ok(const sdr_arb_time_t &s) {
    const u128 v = to_u128(s);
    return v >= ARB_MIN_STEP && v <= ARB_MAX_STEP;
}

}  // namespace

struct ArbHost {
    int dev = 0;
    size_t C = 0;
    std::vector<ArbChan> chans;
    std::vector<float2> tab;                   // every (h, d) table
    size_t hist_len = 0;                       // sum of H_k
    std::vector<u128> step0, first0;           // creation steps and first positions (units of 2^-64 frames)
    // time base: tau(r) = base[k] + (r - rbase[k]) step[k] for r >= rbase[k]
    std::vector<u128> step, base;
    std::vector<unsigned long long> rbase;
    std::vector<unsigned long long> total;     // frames seen, per channel
};

struct sdr_arb : ArbHost {
    StreamRef stream;
    DevBuf d_tab, d_chans, d_call, d_hist[2];
    int cur = 0;
    std::vector<char> call_host;               // tile0 (C + 1) then C ArbCall, uploaded once per call
    DevBuf d_in, d_out;

    int alloc(void *user_stream, const sdr_arb *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_tab.upload(tab.data(), tab.size() * sizeof(float2), stream.s))) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(ArbChan), stream.s))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(hist_len, 1) * 8))) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_arb &src) {
        if (hist_len == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, hist_len * 8, cudaMemcpyDeviceToDevice));
    }
};

// outputs released after n frames in total: #{r >= rbase : tau(r) < n} on top of rbase
static u128 arb_released(const ArbHost &h, size_t k, unsigned long long n) {
    const u128 x = (u128)n << 64;
    if (x <= h.base[k]) return h.rbase[k];
    return (u128)h.rbase[k] + (x - h.base[k] + h.step[k] - 1) / h.step[k];
}

extern "C" int sdr_arb_step(double rate_in, double rate_out, sdr_arb_time_t *step) {
    if (!step) return SDR_ERR_BAD_DATA_PTR;
    if (!(rate_in > 0.0) || !(rate_out > 0.0) || !std::isfinite(rate_in) || !std::isfinite(rate_out))
        return SDR_ERR_INVALID_ARG;
    // rate = m 2^e with 2^52 <= m < 2^53, so rate_in / rate_out = (m1 / m2) 2^(e1 - e2) with m1 / m2 in (1/2, 2)
    int e1, e2;
    const unsigned long long m1 = (unsigned long long)std::ldexp(std::frexp(rate_in, &e1), 53);
    const unsigned long long m2 = (unsigned long long)std::ldexp(std::frexp(rate_out, &e2), 53);
    const long long s = (long long)e1 - e2 + 64;  // the step in units of 2^-64 is (m1 / m2) 2^s
    if (s < 47 || s > 89) return SDR_ERR_INVALID_ARG;  // below 2^-16 or above 2^24 whatever the rounding
    // q = floor(m1 2^s / m2) by long division, r the remainder; then round to nearest, ties to even
    u128 q = m1 / m2;
    unsigned long long r = m1 % m2;
    for (long long i = 0; i < s; ++i) {
        r <<= 1;  // r < m2 < 2^53
        q <<= 1;
        if (r >= m2) {
            r -= m2;
            q |= 1;
        }
    }
    if (2 * r > m2 || (2 * r == m2 && (q & 1))) ++q;
    if (q < ARB_MIN_STEP || q > ARB_MAX_STEP) return SDR_ERR_INVALID_ARG;
    step->whole = (unsigned long long)(q >> 64);
    step->frac = (unsigned long long)q;
    return SDR_OK;
}

extern "C" sdr_arb_t *sdr_arb_create(const sdr_arb_config_t *cfg, int *err) {
    bool ok = cfg && cfg->taps && cfg->step && cfg->n_taps >= 1 && cfg->n_taps <= ARB_MAX_TAPS &&
              cfg->phases >= 1 && cfg->phases <= ARB_MAX_P && (cfg->phases & (cfg->phases - 1)) == 0 &&
              cfg->n_channels >= 1 && cfg->n_channels <= ARB_MAX_CH &&
              (cfg->n_tap_sets == 1 || cfg->n_tap_sets == cfg->n_channels) &&
              cfg->n_tap_sets * cfg->n_taps <= ARB_MAX_TAP_FLOATS;
    for (size_t k = 0; ok && k < cfg->n_channels; ++k)
        ok = step_ok(cfg->step[k]) && (!cfg->first || cfg->first[k].whole < ARB_MAX_POS);
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_arb>(err, cfg->device, cfg->stream, [&](sdr_arb &h) {
        const size_t C = cfg->n_channels, L = cfg->n_taps, P = cfg->phases;
        int p = 0;
        while (((size_t)1 << p) < P) ++p;
        h.C = C;
        h.chans.resize(C);
        h.total.assign(C, 0);
        h.rbase.assign(C, 0);
        h.step0.resize(C);
        h.first0.resize(C);
        // one (h, d) table per distinct tap set
        std::map<size_t, long long> tables;
        for (size_t k = 0; k < C; ++k) {
            const size_t set = cfg->n_tap_sets == 1 ? 0 : k;
            ArbChan &ch = h.chans[k];
            ch.L = (int)L;
            ch.H = (int)((L + P - 1) / P);
            ch.p = p;
            ch.pad = 0;
            ch.hist = (long long)h.hist_len;
            h.hist_len += (size_t)ch.H;
            auto it = tables.find(set);
            if (it == tables.end()) {
                const float *src = cfg->taps + set * L;
                it = tables.emplace(set, (long long)h.tab.size()).first;
                for (size_t j = 0; j < L; ++j) {
                    const double next = j + 1 < L ? (double)src[j + 1] : 0.0;
                    h.tab.push_back(make_float2(src[j], (float)(next - (double)src[j])));
                }
            }
            ch.tab = it->second;
            h.step0[k] = to_u128(cfg->step[k]);
            h.first0[k] = cfg->first ? to_u128(cfg->first[k]) : 0;
        }
        h.step = h.step0;
        h.base = h.first0;
        return SDR_OK;
    });
}

extern "C" void sdr_arb_destroy(sdr_arb_t *h) { destroy_handle(h); }

extern "C" int sdr_arb_reset(sdr_arb_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // frames before the stream read as zero, so the stale history is never used
    std::fill(h->total.begin(), h->total.end(), 0ull);
    std::fill(h->rbase.begin(), h->rbase.end(), 0ull);
    h->step = h->step0;
    h->base = h->first0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_arb_t *sdr_arb_clone(const sdr_arb_t *src, int *err) { return clone_handle<ArbHost>(src, err); }

extern "C" int sdr_arb_set_steps(sdr_arb_t *h, const sdr_arb_time_t *steps) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!steps) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k)
        if (!step_ok(steps[k])) return SDR_ERR_INVALID_ARG;
    for (size_t k = 0; k < h->C; ++k) {
        // the next unreleased output R keeps its position; the new step applies from there on
        const u128 R = arb_released(*h, k, h->total[k]);
        h->base[k] += (R - h->rbase[k]) * h->step[k];
        h->rbase[k] = (unsigned long long)R;
        h->step[k] = to_u128(steps[k]);
    }
    return SDR_OK;
}

extern "C" int sdr_arb_output_count(const sdr_arb_t *h, const size_t *n_in, size_t *counts) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !counts) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) {
        if (n_in[k] > ARB_MAX_POS - 1 - h->total[k]) return SDR_ERR_INVALID_ARG;
        const u128 c = arb_released(*h, k, h->total[k] + n_in[k]) - arb_released(*h, k, h->total[k]);
        if (c >= ARB_MAX_POS) return SDR_ERR_INVALID_ARG;
        counts[k] = (size_t)c;
    }
    return SDR_OK;
}

// in: C device rows (row stride in_stride), row k of n_in[k] frames; out: C rows of out_stride, cnt[k] outputs each
static int arb_run(sdr_arb *h, const float2 *in, const size_t *n_in, size_t in_stride, const size_t *cnt, float2 *out,
                   size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    h->call_host.resize((C + 1) * sizeof(long long) + C * sizeof(ArbCall));
    long long *tile0 = (long long *)h->call_host.data();
    ArbCall *calls = (ArbCall *)(tile0 + C + 1);
    long long tiles = 0;
    bool any = false;
    for (size_t k = 0; k < C; ++k) {
        const unsigned long long T = h->total[k];
        // the call's first output R0 sits at tau(R0) >= T frames
        const u128 R0 = arb_released(*h, k, T);
        const u128 anchor = h->base[k] + (R0 - h->rbase[k]) * h->step[k] - ((u128)T << 64);
        ArbCall &cl = calls[k];
        cl.aw = (unsigned long long)(anchor >> 64);
        cl.af = (unsigned long long)anchor;
        cl.sw = (unsigned long long)(h->step[k] >> 64);
        cl.sf = (unsigned long long)h->step[k];
        cl.cnt = (long long)cnt[k];
        cl.n = (long long)n_in[k];
        cl.lo = -(long long)std::min<unsigned long long>((unsigned long long)h->chans[k].H, T);
        cl.pad = 0;
        any = any || n_in[k] > 0;
        tile0[k] = tiles;
        tiles += (cl.cnt + ARB_THREADS - 1) / ARB_THREADS;
    }
    tile0[C] = tiles;
    if (!any) return SDR_OK;
    int rc = h->d_call.reserve(h->call_host.size());
    if (rc) return rc;
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_call.p, h->call_host.data(), h->call_host.size(), cudaMemcpyHostToDevice, st));
    const long long *d_tile0 = (const long long *)h->d_call.p;
    const ArbCall *d_calls = (const ArbCall *)(d_tile0 + C + 1);
    const long long stride = C > 1 ? (long long)in_stride : 0;
    if (tiles > 0) {
        const unsigned grid = (unsigned)std::min<long long>(tiles, 1LL << 30);
        arb_kernel<<<grid, ARB_THREADS, 0, st>>>((const float2 *)h->d_tab.p, (const ArbChan *)h->d_chans.p, d_calls,
                                                 d_tile0, (int)C, tiles, (const float2 *)h->d_hist[h->cur].p, in,
                                                 stride, out, (long long)out_stride);
        count_launch();
        if ((rc = launch_status())) return rc;
    }
    arb_carry_kernel<<<(unsigned)C, ARB_THREADS, 0, st>>>((const ArbChan *)h->d_chans.p, d_calls,
                                                          (const float2 *)h->d_hist[h->cur].p, in, stride,
                                                          (float2 *)h->d_hist[h->cur ^ 1].p);
    count_launch();
    if ((rc = launch_status())) return rc;
    h->cur ^= 1;
    for (size_t k = 0; k < C; ++k) h->total[k] += n_in[k];
    return SDR_OK;
}

static int arb_check(const sdr_arb *h, const float *in, const size_t *n_in, size_t in_stride, const float *out,
                     size_t out_cap, size_t out_stride, size_t *n_out, std::vector<size_t> &cnt, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out || !n_in) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = 0;
    *longest = *std::max_element(n_in, n_in + h->C);
    if (*longest > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < *longest) return SDR_ERR_INVALID_ARG;
    cnt.resize(h->C);
    int rc = sdr_arb_output_count(h, n_in, cnt.data());
    if (rc) return rc;
    const size_t most = *std::max_element(cnt.begin(), cnt.end());
    if (most > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (most > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (most > 0 && h->C > 1 && out_stride < most) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_arb_process_dev(sdr_arb_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                   float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    size_t longest = 0;
    int rc = arb_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, cnt, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = arb_run(h, (const float2 *)in_c64, n_in, in_stride, cnt.data(), (float2 *)out_c64, out_stride);
    if (rc) return rc;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = cnt[k];
    return SDR_OK;
}

extern "C" int sdr_arb_process(sdr_arb_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                               float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    size_t longest = 0;
    int rc = arb_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, cnt, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t stride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : out_cap;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` frames per channel: H2D, compute, D2H in stream order
    const size_t chunk = std::min(longest, std::max<size_t>(1, ARB_HOST_BYTES / (C * 8)));
    const bool equal_in = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    std::vector<size_t> take(C), part(C), done(C, 0);
    size_t fcap = 1;
    for (size_t k = 0; k < C; ++k) {  // a chunk releases at most ceil(chunk / sigma) outputs
        const u128 lim = (((u128)chunk << 64) + h->step[k] - 1) / h->step[k];
        fcap = std::max<size_t>(fcap, (size_t)std::min<u128>(lim, cnt[k]));
    }
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
        if ((rc = sdr_arb_output_count(h, take.data(), part.data()))) return rc;
        rc = arb_run(h, (const float2 *)h->d_in.p, take.data(), chunk, part.data(), (float2 *)h->d_out.p, fcap);
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

// tsync.cu -- K15, sdr_tsync_*: symbol timing recovery bank.  C independent c64 channel streams; channel k has real
// taps h_k of length L at P = 2^p times the input rate (sdr_arb's interpolant A(t), bit for bit: arb_core.cuh), a
// nominal symbol period T in units of 2^-64 frames, a first on-time position tau(0) and a Gardner loop
// {kp, ki, err_max, max_dev}.  Loop quantities are int64 in units of 2^-40 frames, q(x) = rint(x 2^40) for an f32 x,
// V = floor(max_dev T) in those units.  With v_0 = 0, y_{-1} = 0, for s = 0, 1, ...:
//     T_s = T + 2^24 v_s,  y_s = A(tau_s),  m_s = A(tau_s - floor(T_s / 2))  (s >= 1)
//     g = fl(fl(fl(y_s.re - y_{s-1}.re) m_s.re) + fl(fl(y_s.im - y_{s-1}.im) m_s.im))
//     e_s = 0 for s = 0 or a non-finite g, else min(max(g, -err_max), err_max)
//     v_{s+1} = clamp(v_s - q(fl(ki e_s)), -V, V)
//     tau_{s+1} = tau_s + T + 2^24 v_{s+1} - 2^24 q(fl(kp e_s))
// Every f32 operation of the loop is rounded on its own (__fsub_rn / __fmul_rn / __fadd_rn: nothing is contracted).
// Symbol s is released by the first call after which the channel's frame total n satisfies floor(tau_s) < n.
// The loop is a recurrence: one thread runs one channel's symbols in order, and the positions, v and y_{s-1} of every
// channel live on the device between calls, so a call's counts are copied back before it returns.
// Carried across calls: the last ceil(L / P) + ceil((T + V) / 2) + 1 frames of every channel and its frame total.
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
typedef __int128 i128;

constexpr size_t TS_MAX_CH = 65536;
constexpr size_t TS_MAX_TAPS = (size_t)1 << 20;
constexpr size_t TS_MAX_TAP_FLOATS = (size_t)1 << 26;
constexpr size_t TS_MAX_P = (size_t)1 << 16;
constexpr u128 TS_MIN_PERIOD = (u128)1 << 64;           // 1 frame
constexpr u128 TS_MAX_PERIOD = (u128)1 << 84;           // 2^20 frames
constexpr unsigned long long TS_MAX_POS = 1ull << 62;  // whole parts, frame totals and per-call counts stay below
constexpr int TS_THREADS = 32;                          // one channel per thread; one warp per CTA spreads channels
constexpr size_t TS_HOST_BYTES = (size_t)32 << 20;     // host-memory calls: chunk size of input

struct TsChan {                  // per channel, fixed at create
    long long tab;               // offset (float2 entries) of the channel's (h, d) table
    long long hist;              // offset of the channel's Hc carried frames in a history buffer
    int L, p, Hc, pad;           // taps, log2 P, carried frames
    unsigned long long tw, tf;   // nominal period T (whole, fraction)
    long long V;                 // bound of |v|, 2^-40 frames
    float kp, ki, emax, pad2;
};

struct TsState {                 // per channel, on the device between calls
    unsigned long long tw, tf;   // tau of the next unreleased symbol (absolute)
    long long v;                 // period offset, 2^-40 frames
    float2 yprev;                // y_{s-1}
    unsigned long long nsym;     // symbols released so far
};

struct TsCall {                  // per channel and call
    long long base;              // frames before the call
    long long n;                 // frames of the call
    long long lo;                // frames (relative to the call) below lo lie before the stream and read as 0
    long long cap;               // the call's bound on its symbols
};

// y = A(on-time position), m = A(mid position): sdr_arb's chains (arb_core.cuh) with their terms interleaved.  The two
// positions are split into frame (relative to the call), phase and truncated weight exactly as arb_kernel does.
template <bool CHECK>
__device__ __forceinline__ void ts_pair(const float2 *__restrict__ tab, int L, int p, long long ny,
                                        unsigned long long fy, long long nm, unsigned long long fm, const float2 *hist,
                                        const float2 *y, long long lo, float2 &zy, float2 &zm) {
    const int P = 1 << p;
    const int ipy = p ? (int)(fy >> (64 - p)) : 0, ipm = p ? (int)(fm >> (64 - p)) : 0;
    const float ay = (float)((fy << p) >> 40) * 0x1p-24f, am = (float)((fm << p) >> 40) * 0x1p-24f;
    const int Ty = ipy < L ? ((L - ipy + P - 1) >> p) : 0, Tm = ipm < L ? ((L - ipm + P - 1) >> p) : 0;
    const float2 *tby = tab + ipy, *tbm = tab + ipm;
    zy = make_float2(0.f, 0.f);
    zm = make_float2(0.f, 0.f);
    const int Tc = min(Ty, Tm);
#pragma unroll 2
    for (int i = 0; i < Tc; ++i) {
        const float2 hy = __ldg(tby + (long long)i * P), hm = __ldg(tbm + (long long)i * P);
        const float cy = arb_tap(hy, ay), cm = arb_tap(hm, am);
        const float2 vy = CHECK ? arb_load(hist, y, ny - i, lo) : __ldg(y + (ny - i));
        const float2 vm = CHECK ? arb_load(hist, y, nm - i, lo) : __ldg(y + (nm - i));
        arb_acc(cy, vy, zy);
        arb_acc(cm, vm, zm);
    }
    for (int i = Tc; i < Ty; ++i)  // the two term counts differ by at most one
        arb_acc(arb_tap(__ldg(tby + (long long)i * P), ay), arb_load(hist, y, ny - i, lo), zy);
    for (int i = Tc; i < Tm; ++i)
        arb_acc(arb_tap(__ldg(tbm + (long long)i * P), am), arb_load(hist, y, nm - i, lo), zm);
}

// q(x) = rint(x 2^40) for an f32 x (|x| < 2^22: the scaling is exact and the result fits)
__device__ __forceinline__ long long ts_q(float x) { return __float2ll_rn(__fmul_rn(x, 0x1p40f)); }

// One thread per channel runs its symbols in order until the next on-time position lies past the call's frames.
__global__ void __launch_bounds__(TS_THREADS) tsync_kernel(const float2 *__restrict__ tab,
                                                           const TsChan *__restrict__ chans,
                                                           const TsCall *__restrict__ calls, TsState *state, int C,
                                                           const float2 *__restrict__ hist,
                                                           const float2 *__restrict__ in, long long in_stride,
                                                           float2 *__restrict__ sym, sdr_arb_time_t *__restrict__ pos,
                                                           float *__restrict__ err, long long out_stride,
                                                           long long *__restrict__ counts) {
    const int k = blockIdx.x * TS_THREADS + threadIdx.x;
    if (k >= C) return;
    const TsChan ch = chans[k];
    const TsCall cl = calls[k];
    TsState st = state[k];
    const float2 *y = in + k * in_stride;
    const float2 *hk = hist + ch.hist + ch.Hc;
    const float2 *tb = tab + ch.tab;
    const u128 T = ((u128)ch.tw << 64) | ch.tf;
    const u128 end = (u128)(unsigned long long)(cl.base + cl.n) << 64;
    const long long rows = k * out_stride;
    u128 tau = ((u128)st.tw << 64) | st.tf;
    long long v = st.v, cnt = 0;
    float2 yp = st.yprev;
    while (tau < end && cnt < cl.cap) {
        // mid position tau - floor(T_s / 2) for s >= 1 (it lies at or after tau_{s-1}); symbol 0 reads tau twice
        const u128 Ts = (u128)((i128)T + ((i128)v << 24));
        const u128 mid = st.nsym ? tau - (Ts >> 1) : tau;
        const long long ny = (long long)(unsigned long long)(tau >> 64) - cl.base;
        const long long nm = (long long)(unsigned long long)(mid >> 64) - cl.base;
        float2 zy, zm;
        if (nm - ch.Hc >= 0)
            ts_pair<false>(tb, ch.L, ch.p, ny, (unsigned long long)tau, nm, (unsigned long long)mid, hk, y, cl.lo, zy,
                           zm);
        else
            ts_pair<true>(tb, ch.L, ch.p, ny, (unsigned long long)tau, nm, (unsigned long long)mid, hk, y, cl.lo, zy,
                          zm);
        float e = 0.f;
        if (st.nsym) {
            const float g = __fadd_rn(__fmul_rn(__fsub_rn(zy.x, yp.x), zm.x), __fmul_rn(__fsub_rn(zy.y, yp.y), zm.y));
            if (isfinite(g)) e = fminf(fmaxf(g, -ch.emax), ch.emax);
        }
        sym[rows + cnt] = zy;
        if (pos) pos[rows + cnt] = sdr_arb_time_t{(unsigned long long)(tau >> 64), (unsigned long long)tau};
        if (err) err[rows + cnt] = e;
        const long long v1 = min(max(v - ts_q(__fmul_rn(ch.ki, e)), -ch.V), ch.V);
        tau += (u128)((i128)T + ((i128)(v1 - ts_q(__fmul_rn(ch.kp, e))) << 24));
        v = v1;
        yp = zy;
        ++st.nsym;
        ++cnt;
    }
    st.tw = (unsigned long long)(tau >> 64);
    st.tf = (unsigned long long)tau;
    st.v = v;
    st.yprev = yp;
    state[k] = st;
    counts[k] = cnt;
}

// history: the last Hc frames of (carried frames, the call's row), per channel; one CTA per channel
__global__ void __launch_bounds__(128) tsync_carry_kernel(const TsChan *__restrict__ chans,
                                                          const TsCall *__restrict__ calls,
                                                          const float2 *__restrict__ hist_old,
                                                          const float2 *__restrict__ in, long long in_stride,
                                                          float2 *__restrict__ hist_new) {
    const int k = blockIdx.x;
    const TsChan ch = chans[k];
    bank_carry(hist_old, in + k * in_stride, calls[k].n, ch.Hc, ch.hist, hist_new);
}

u128 to_u128(const sdr_arb_time_t &t) { return ((u128)t.whole << 64) | t.frac; }

// q(x) on the host, for |x| < 2^22
long long q40(float x) { return std::llrint((double)x * 0x1p40); }

// floor(max_dev T) in units of 2^-40 frames, T in units of 2^-64, from max_dev's binary value: max_dev = m 2^(e-53),
// so V = floor(m T / 2^(77 - e)) with 77 - e >= 78 for max_dev <= 0.25; m T = A 2^64 + B with B < 2^64 gives
// V = floor(A / 2^(13 - e)).
long long dev_bound(double max_dev, u128 T) {
    if (max_dev == 0.0) return 0;
    int e = 0;
    const unsigned long long m = (unsigned long long)std::ldexp(std::frexp(max_dev, &e), 53);
    const u128 lo = (u128)m * (unsigned long long)T;
    const u128 A = (u128)m * (unsigned long long)(T >> 64) + (lo >> 64);
    const int sh = 13 - e;
    return sh >= 128 ? 0 : (long long)(A >> sh);
}

}  // namespace

struct TsyncHost {
    int dev = 0;
    size_t C = 0;
    std::vector<TsChan> chans;
    std::vector<float2> tab;                  // every (h, d) table
    size_t hist_len = 0;                      // sum of Hc
    std::vector<TsState> init;                // the creation state
    std::vector<u128> tmin;                   // T - 2^24 V - 2^24 q(fl(kp err_max)): the least step
    std::vector<unsigned long long> total;    // frames seen, per channel
    bool fresh = true;                        // the device state is the creation state's once uploaded
};

struct sdr_tsync : TsyncHost {
    StreamRef stream;
    DevBuf d_tab, d_chans, d_call, d_state, d_hist[2];
    int cur = 0;
    std::vector<TsCall> call_host;
    std::vector<long long> cnt_host;
    DevBuf d_in, d_sym, d_pos, d_err;

    int alloc(void *user_stream, const sdr_tsync *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_tab.upload(tab.data(), tab.size() * sizeof(float2), stream.s))) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(TsChan), stream.s))) return rc;
        if ((rc = d_state.alloc(C * sizeof(TsState)))) return rc;
        if ((rc = d_call.alloc(C * (sizeof(TsCall) + sizeof(long long))))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(hist_len, 1) * 8))) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_tsync &src) {
        SDR_CUDA_TRY(cudaMemcpy(d_state.p, src.d_state.p, C * sizeof(TsState), cudaMemcpyDeviceToDevice));
        if (hist_len == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, hist_len * 8, cudaMemcpyDeviceToDevice));
    }
};

extern "C" int sdr_tsync_loop_design(double bn_t, double zeta, double ted_gain, double period_frames, float *kp,
                                     float *ki) {
    if (!kp || !ki) return SDR_ERR_BAD_DATA_PTR;
    for (double x : {bn_t, zeta, ted_gain, period_frames})
        if (!(x > 0.0) || !std::isfinite(x)) return SDR_ERR_INVALID_ARG;
    const double th = bn_t / (zeta + 1.0 / (4.0 * zeta));
    const double d = 1.0 + 2.0 * zeta * th + th * th;
    *kp = (float)(4.0 * zeta * th / (d * ted_gain) * period_frames);
    *ki = (float)(4.0 * th * th / (d * ted_gain) * period_frames);
    return SDR_OK;
}

extern "C" sdr_tsync_t *sdr_tsync_create(const sdr_tsync_config_t *cfg, int *err) {
    bool ok = cfg && cfg->taps && cfg->period && cfg->loops && cfg->n_taps >= 1 && cfg->n_taps <= TS_MAX_TAPS &&
              cfg->phases >= 1 && cfg->phases <= TS_MAX_P && (cfg->phases & (cfg->phases - 1)) == 0 &&
              cfg->n_channels >= 1 && cfg->n_channels <= TS_MAX_CH &&
              (cfg->n_tap_sets == 1 || cfg->n_tap_sets == cfg->n_channels) &&
              cfg->n_tap_sets * cfg->n_taps <= TS_MAX_TAP_FLOATS &&
              (cfg->n_loops == 1 || cfg->n_loops == cfg->n_channels);
    std::vector<long long> V, D;
    for (size_t k = 0; ok && k < cfg->n_channels; ++k) {
        const sdr_tsync_loop_t &lp = cfg->loops[cfg->n_loops == 1 ? 0 : k];
        const u128 T = to_u128(cfg->period[k]);
        ok = T >= TS_MIN_PERIOD && T <= TS_MAX_PERIOD && (!cfg->first || cfg->first[k].whole < TS_MAX_POS) &&
             lp.max_dev >= 0.0 && lp.max_dev <= 0.25 && lp.kp >= 0.f && lp.ki >= 0.f && std::isfinite(lp.kp) &&
             std::isfinite(lp.ki) && lp.err_max > 0.f && std::isfinite(lp.err_max);
        if (!ok) break;
        const float pe = lp.kp * lp.err_max, ie = lp.ki * lp.err_max;
        ok = ie < 0x1p22f && pe < 0x1p22f;
        if (!ok) break;
        V.push_back(dev_bound(lp.max_dev, T));
        D.push_back(q40(pe));
        // 2 D < T - V (all in units of 2^-64): steps stay above T - V - D > 0, mid samples after the previous symbol
        ok = ((u128)2 * ((u128)D.back() << 24)) < T - ((u128)V.back() << 24);
    }
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_tsync>(err, cfg->device, cfg->stream, [&](sdr_tsync &h) {
        const size_t C = cfg->n_channels, L = cfg->n_taps, P = cfg->phases;
        int p = 0;
        while (((size_t)1 << p) < P) ++p;
        h.C = C;
        h.chans.resize(C);
        h.init.resize(C);
        h.tmin.resize(C);
        h.total.assign(C, 0);
        std::map<size_t, long long> tables;
        for (size_t k = 0; k < C; ++k) {
            const size_t set = cfg->n_tap_sets == 1 ? 0 : k;
            const sdr_tsync_loop_t &lp = cfg->loops[cfg->n_loops == 1 ? 0 : k];
            const u128 T = to_u128(cfg->period[k]);
            TsChan &ch = h.chans[k];
            ch.L = (int)L;
            ch.p = p;
            // ceil(L / P) frames for a chain, ceil((T + V) / 2) more for the mid position, one for its floor
            const u128 half = (T + ((u128)V[k] << 24) + ((u128)1 << 65) - 1) >> 65;
            ch.Hc = (int)((L + P - 1) / P + (size_t)half + 1);
            ch.pad = 0;
            ch.hist = (long long)h.hist_len;
            h.hist_len += (size_t)ch.Hc;
            ch.tw = (unsigned long long)(T >> 64);
            ch.tf = (unsigned long long)T;
            ch.V = V[k];
            ch.kp = lp.kp;
            ch.ki = lp.ki;
            ch.emax = lp.err_max;
            ch.pad2 = 0.f;
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
            const sdr_arb_time_t f0 = cfg->first ? cfg->first[k] : sdr_arb_time_t{0, 0};
            h.init[k] = TsState{f0.whole, f0.frac, 0, make_float2(0.f, 0.f), 0};
            h.tmin[k] = T - ((u128)V[k] << 24) - ((u128)D[k] << 24);
        }
        return SDR_OK;
    });
}

extern "C" void sdr_tsync_destroy(sdr_tsync_t *h) { destroy_handle(h); }

extern "C" int sdr_tsync_reset(sdr_tsync_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // the next call uploads the creation state; frames before the stream read as zero, so stale history is unused
    std::fill(h->total.begin(), h->total.end(), 0ull);
    h->fresh = true;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_tsync_t *sdr_tsync_clone(const sdr_tsync_t *src, int *err) { return clone_handle<TsyncHost>(src, err); }

extern "C" int sdr_tsync_max_output(const sdr_tsync_t *h, const size_t *n_in, size_t *caps) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !caps) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) {
        if (n_in[k] > TS_MAX_POS - 1 - h->total[k]) return SDR_ERR_INVALID_ARG;
        // unreleased positions lie at or after the frame total and steps are at least tmin
        caps[k] = (size_t)((((u128)n_in[k] << 64) + h->tmin[k] - 1) / h->tmin[k]);
    }
    return SDR_OK;
}

extern "C" int sdr_tsync_get_state(sdr_tsync_t *h, size_t channel, sdr_arb_time_t *next, int64_t *v) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!next || !v) return SDR_ERR_BAD_DATA_PTR;
    if (channel >= h->C) return SDR_ERR_INVALID_ARG;
    TsState st = h->init[channel];
    if (!h->fresh) {
        DeviceGuard g(h->dev);
        if (!g.ok) return g.status();
        SDR_CUDA_TRY(cudaMemcpyAsync(&st, (const TsState *)h->d_state.p + channel, sizeof(TsState),
                                     cudaMemcpyDeviceToHost, h->stream.s));
        SDR_CUDA_TRY(cudaStreamSynchronize(h->stream.s));
    }
    next->whole = st.tw;
    next->frac = st.tf;
    *v = st.v;
    return SDR_OK;
}

// in: C device rows (row stride in_stride), row k of n_in[k] frames; outputs: C rows of out_stride, at most cap[k]
// symbols each.  Returns once the counts are on the host (got).
static int ts_run(sdr_tsync *h, const float2 *in, const size_t *n_in, size_t in_stride, const size_t *cap,
                  float2 *sym, sdr_arb_time_t *pos, float *err, size_t out_stride, size_t *got) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    for (size_t k = 0; k < C; ++k) got[k] = 0;
    if (std::all_of(n_in, n_in + C, [](size_t n) { return n == 0; })) return SDR_OK;
    h->call_host.resize(C);
    h->cnt_host.resize(C);
    for (size_t k = 0; k < C; ++k) {
        const unsigned long long T = h->total[k];
        h->call_host[k] = TsCall{(long long)T, (long long)n_in[k],
                                 -(long long)std::min<unsigned long long>((unsigned long long)h->chans[k].Hc, T),
                                 (long long)cap[k]};
    }
    if (h->fresh) {
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_state.p, h->init.data(), C * sizeof(TsState), cudaMemcpyHostToDevice, st));
        h->fresh = false;
    }
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_call.p, h->call_host.data(), C * sizeof(TsCall), cudaMemcpyHostToDevice, st));
    const TsCall *d_calls = (const TsCall *)h->d_call.p;
    long long *d_cnt = (long long *)(d_calls + C);
    const long long stride = C > 1 ? (long long)in_stride : 0;
    tsync_kernel<<<(unsigned)((C + TS_THREADS - 1) / TS_THREADS), TS_THREADS, 0, st>>>(
        (const float2 *)h->d_tab.p, (const TsChan *)h->d_chans.p, d_calls, (TsState *)h->d_state.p, (int)C,
        (const float2 *)h->d_hist[h->cur].p, in, stride, sym, pos, err, C > 1 ? (long long)out_stride : 0, d_cnt);
    count_launch();
    int rc = launch_status();
    if (rc) return rc;
    tsync_carry_kernel<<<(unsigned)C, 128, 0, st>>>((const TsChan *)h->d_chans.p, d_calls,
                                                    (const float2 *)h->d_hist[h->cur].p, in, stride,
                                                    (float2 *)h->d_hist[h->cur ^ 1].p);
    count_launch();
    if ((rc = launch_status())) return rc;
    h->cur ^= 1;
    for (size_t k = 0; k < C; ++k) h->total[k] += n_in[k];
    SDR_CUDA_TRY(cudaMemcpyAsync(h->cnt_host.data(), d_cnt, C * sizeof(long long), cudaMemcpyDeviceToHost, st));
    SDR_CUDA_TRY(cudaStreamSynchronize(st));
    for (size_t k = 0; k < C; ++k) got[k] = (size_t)h->cnt_host[k];
    return SDR_OK;
}

static int ts_check(const sdr_tsync *h, const float *in, const size_t *n_in, size_t in_stride, const float *sym,
                    size_t out_cap, size_t out_stride, size_t *n_out, std::vector<size_t> &cap, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out || !n_in) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = 0;
    *longest = *std::max_element(n_in, n_in + h->C);
    if (*longest > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < *longest) return SDR_ERR_INVALID_ARG;
    cap.resize(h->C);
    int rc = sdr_tsync_max_output(h, n_in, cap.data());
    if (rc) return rc;
    const size_t most = *std::max_element(cap.begin(), cap.end());
    if (most > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (most > 0 && !sym) return SDR_ERR_BAD_DATA_PTR;
    if (most > 0 && h->C > 1 && out_stride < most) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_tsync_process_dev(sdr_tsync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                     float *sym_c64, sdr_arb_time_t *pos, float *err, size_t out_cap,
                                     size_t out_stride, size_t *n_out) {
    std::vector<size_t> cap;
    size_t longest = 0;
    int rc = ts_check(h, in_c64, n_in, in_stride, sym_c64, out_cap, out_stride, n_out, cap, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)sym_c64 % 8) != 0 || ((uintptr_t)pos % 8) != 0 ||
        ((uintptr_t)err % 4) != 0)
        return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    return ts_run(h, (const float2 *)in_c64, n_in, in_stride, cap.data(), (float2 *)sym_c64, pos, err, out_stride,
                  n_out);
}

extern "C" int sdr_tsync_process(sdr_tsync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                 float *sym_c64, sdr_arb_time_t *pos, float *err, size_t out_cap, size_t out_stride,
                                 size_t *n_out) {
    std::vector<size_t> cap;
    size_t longest = 0;
    int rc = ts_check(h, in_c64, n_in, in_stride, sym_c64, out_cap, out_stride, n_out, cap, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t stride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : out_cap;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` frames per channel: H2D, compute (which returns the counts), D2H
    const size_t chunk = std::min(longest, std::max<size_t>(1, TS_HOST_BYTES / (C * 8)));
    const bool equal_in = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    std::vector<size_t> take(C), ccap(C), part(C), done(C, 0);
    std::vector<size_t> full(C, chunk);
    if ((rc = sdr_tsync_max_output(h, full.data(), ccap.data()))) return rc;
    const size_t fcap = std::max<size_t>(1, *std::max_element(ccap.begin(), ccap.end()));
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_sym.reserve(fcap * C * 8);
    if (!rc && pos) rc = h->d_pos.reserve(fcap * C * sizeof(sdr_arb_time_t));
    if (!rc && err) rc = h->d_err.reserve(fcap * C * 4);
    if (rc) return rc;
    // one array of C rows from the device rows (fcap apart) to the caller's rows (ostride apart) at done[k]
    auto fetch = [&](void *dst, const void *src, size_t bytes) -> int {
        const bool equal = std::all_of(part.begin(), part.end(), [&](size_t p) { return p == part[0]; }) &&
                           std::all_of(done.begin(), done.end(), [&](size_t d) { return d == done[0]; });
        if (equal && part[0] > 0)
            SDR_CUDA_TRY(cudaMemcpy2DAsync((char *)dst + done[0] * bytes, ostride * bytes, src, fcap * bytes,
                                           part[0] * bytes, C, cudaMemcpyDeviceToHost, st));
        else if (!equal)
            for (size_t k = 0; k < C; ++k)
                if (part[k])
                    SDR_CUDA_TRY(cudaMemcpyAsync((char *)dst + (k * ostride + done[k]) * bytes,
                                                 (const char *)src + k * fcap * bytes, part[k] * bytes,
                                                 cudaMemcpyDeviceToHost, st));
        return SDR_OK;
    };
    for (size_t at = 0; at < longest; at += chunk) {
        for (size_t k = 0; k < C; ++k) take[k] = n_in[k] > at ? std::min(chunk, n_in[k] - at) : 0;
        if (equal_in)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, chunk * 8, in_c64 + 2 * at, stride * 8, take[0] * 8, C,
                                           cudaMemcpyHostToDevice, st));
        else
            for (size_t k = 0; k < C; ++k)
                if (take[k])
                    SDR_CUDA_TRY(cudaMemcpyAsync((float2 *)h->d_in.p + k * chunk, in_c64 + 2 * (k * stride + at),
                                                 take[k] * 8, cudaMemcpyHostToDevice, st));
        if ((rc = sdr_tsync_max_output(h, take.data(), ccap.data()))) return rc;
        rc = ts_run(h, (const float2 *)h->d_in.p, take.data(), chunk, ccap.data(), (float2 *)h->d_sym.p,
                    pos ? (sdr_arb_time_t *)h->d_pos.p : nullptr, err ? (float *)h->d_err.p : nullptr, fcap,
                    part.data());
        if (rc) return rc;
        if ((rc = fetch(sym_c64, h->d_sym.p, 8))) return rc;
        if (pos && (rc = fetch(pos, h->d_pos.p, sizeof(sdr_arb_time_t)))) return rc;
        if (err && (rc = fetch(err, h->d_err.p, 4))) return rc;
        for (size_t k = 0; k < C; ++k) done[k] += part[k];
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    for (size_t k = 0; k < C; ++k) n_out[k] = done[k];
    return SDR_OK;
}

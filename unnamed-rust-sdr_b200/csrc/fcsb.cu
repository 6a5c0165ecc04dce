// fcsb.cu -- K12, sdr_fcsb_*: fast-convolution (overlap-save) synthesis bank, the transpose of K9.  sdr_duc's function
// with one interpolation I_k per channel: channel k (frames before the stream 0) is zero-stuffed by I_k on sdr_pfs's
// grid, filtered by real taps h_k, mixed UP by its 64-bit NCO, and all channels are summed; F = first_sample is the
// absolute index of output 0:
//     s_k[(m+1) I_k - 1] = y_k[m],  u_k[n] = sum_{j<L} h_k[j] s_k[n - j],  x[n] = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64}
// computed rotate-first: w_k = s_k e^{+2 pi i phi_k(F + n)} (nonzero only at frames, so the rotation runs at the low
// rate with the exact integer phase), then x = sum_k g_k * w_k with K9's rotated taps g_k[j] = h_k[j] e^{+2 pi i j Delta_k}.
//
// Geometry: K9's (sdr_fcfb_geometry with D = I): Il = lcm(I_k), N, P; block b holds the outputs at absolute indices
// [b P + eps, (b + 1) P + eps), eps = F mod Il, and its span is the N positions ending at its last output.  Il | P puts
// channel k's frames at the same span positions t = rho_k + i I_k in every block, rho_k = (N - P - 1) mod I_k.
//
// Per slab of whole blocks (about 32 MiB of spectra):
//   fcsb_gather_kernel   v_kb[u] = w_k at span position g_k u + rho_k (u < M_k = N / g_k, g_k = the largest power of
//                        two dividing I_k): the rotated frame where u is a multiple of I_k / g_k, 0 elsewhere and past
//                        the span; frames read through (carried frames, caller's row) pointers; rows grouped by M_k
//   sdr_fft plans M_k    V_kb = DFT_{M_k}(v_kb), one plan per distinct M_k
//   fcsb_unfold_kernel   conj(S_b[r]), S_b[r] = sum_k G'_k[r] V_kb[r mod M_k], k ascending, G'_k[r] = DFT_N(g_k)[r]
//                        e^{-2 pi i r rho_k / N} (host f64, rounded to f32 once)
//   sdr_fft plan N       the inverse through conjugation, IDFT(S) = conj(DFT(conj S)) / N
//   fcsb_store_kernel    the last P positions of each block, (1/N) conj(.), into the caller's contiguous output
// The rotation is K9's: one f64 sincospi of the exact integer phase per (block, channel, run of 1024 frames) times a
// per-channel f32 table.  Every output depends only on its block's span and its absolute position, so blockings,
// clones and block-aligned primed shards give the same bits.
#include <algorithm>
#include <climits>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "nco.cuh"

using namespace sdr;

namespace {

constexpr size_t FCSB_MAX_CH = 256;
constexpr size_t FCSB_MAX_TAPS = (size_t)1 << 20;
constexpr size_t FCSB_SLAB_BYTES = (size_t)32 << 20;  // c64 spectra of one slab (a few waves of the N-point plan)
constexpr size_t FCSB_ROWS_BYTES = (size_t)128 << 20; // at most this much of unfold rows per slab
constexpr size_t FCSB_HOST_BYTES = (size_t)32 << 20;  // host-memory calls: input and output chunk size
constexpr int FCSB_RUN = 1024;                        // frames per rotation base (table length)
constexpr int FCSB_UNFOLD_BLOCKS = 4;                 // blocks per unfold thread (G' read once for all of them)

struct FcsbChan {
    long long M;       // small transform size N / g
    long long us;      // I / g: frames sit at multiples of us in v
    long long I;
    long long rho;     // span position of the first frame
    long long nfr;     // frames in a span: ceil((N - rho) / I)
    long long base;    // rows of this channel start at slab offset B * base (units of c64)
    long long fpb;     // frames per block P / I
    long long fr0;     // handle frame index of block j's first span frame = (j + 1) fpb + fr0
    long long fil;     // Il / I
    uint64_t inc;
};

// Frame m of channel k in one call: 0 for m < 0, hist[k hs + m - hq fil_k] below iq fil_k (the carried frames), then
// in[k is + m - iq fil_k] (the caller's row, never copied); hq, iq are the handle positions of the carried frames and
// of the call's first frame, divided by Il
struct FcsbSrc {
    const float2 *hist;
    const float2 *in;
    long long hs, is;
    long long hq, iq;
};

__device__ __forceinline__ float2 fcsb_load(const FcsbSrc &s, int k, long long fil, long long m) {
    if (m < 0) return make_float2(0.f, 0.f);
    const long long i0 = s.iq * fil;
    if (m < i0) return __ldg(s.hist + k * s.hs + (m - s.hq * fil));
    return __ldg(s.in + k * s.is + (m - i0));
}

// CTA = (256 bins u of channel blockIdx.y, block blockIdx.z of the slab).  The rotation of frame i of block j is
// base(run i / FCSB_RUN) tab[k][i mod FCSB_RUN], base = e^{+2 pi i A Delta_k / 2^64} at the run's first frame, A its
// absolute index F + (m + 1) I - 1; a CTA's frames touch at most two runs.
__global__ void __launch_bounds__(256) fcsb_gather_kernel(FcsbSrc src, const FcsbChan *__restrict__ chan,
                                                          const float2 *__restrict__ tab, long long N, long long nb,
                                                          long long j0, uint64_t first, float2 *__restrict__ v) {
    __shared__ float2 base_s[2];
    const int k = blockIdx.y;
    const FcsbChan c = chan[k];
    const long long u0 = (long long)blockIdx.x * blockDim.x;
    if (u0 >= c.M) return;
    const long long b = blockIdx.z, u = u0 + threadIdx.x;
    const long long m0 = (j0 + b + 1) * c.fpb + c.fr0;  // handle frame of span frame 0
    const long long run0 = (u0 / c.us) / FCSB_RUN;
    if (threadIdx.x < 2) {
        const long long m = m0 + (run0 + threadIdx.x) * FCSB_RUN;
        const float2 r = nco_rot((first + (uint64_t)((m + 1) * c.I - 1)) * c.inc);
        base_s[threadIdx.x] = make_float2(r.x, -r.y);
    }
    __syncthreads();
    if (u >= c.M) return;
    float2 w = make_float2(0.f, 0.f);
    const long long i = u / c.us;
    if (u == i * c.us && i < c.nfr) {
        const float2 y = fcsb_load(src, k, c.fil, m0 + i);
        const float2 rt = cmul(base_s[i / FCSB_RUN - run0], __ldg(tab + (size_t)k * FCSB_RUN + (i % FCSB_RUN)));
        w = cmul(rt, y);
    }
    v[nb * c.base + b * c.M + u] = w;
}

// thread = (bin r < N, FCSB_UNFOLD_BLOCKS blocks): conj(sum_k G'_k[r] V_kb[r mod M_k]), k ascending
__global__ void __launch_bounds__(256) fcsb_unfold_kernel(const float2 *__restrict__ V, const float2 *__restrict__ G,
                                                          const longlong2 *__restrict__ mb, int C, long long N,
                                                          long long nb, float2 *__restrict__ S) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= N) return;
    const long long b0 = (long long)blockIdx.y * FCSB_UNFOLD_BLOCKS;
    const int nq = (int)min((long long)FCSB_UNFOLD_BLOCKS, nb - b0);
    float ar[FCSB_UNFOLD_BLOCKS], ai[FCSB_UNFOLD_BLOCKS];
#pragma unroll
    for (int q = 0; q < FCSB_UNFOLD_BLOCKS; ++q) ar[q] = ai[q] = 0.f;
    for (int k = 0; k < C; ++k) {
        const longlong2 c = __ldg(mb + k);  // (M_k, base_k)
        const float2 w = __ldg(G + (size_t)k * N + r);
        const float2 *Vk = V + nb * c.y + b0 * c.x + (r & (c.x - 1));
#pragma unroll
        for (int q = 0; q < FCSB_UNFOLD_BLOCKS; ++q) {
            if (q < nq) {
                const float2 x = __ldg(Vk + q * c.x);
                ar[q] = __fmaf_rn(w.x, x.x, ar[q]);
                ar[q] = __fmaf_rn(-w.y, x.y, ar[q]);
                ai[q] = __fmaf_rn(w.x, x.y, ai[q]);
                ai[q] = __fmaf_rn(w.y, x.x, ai[q]);
            }
        }
    }
    float2 *Sb = S + b0 * N + r;
#pragma unroll
    for (int q = 0; q < FCSB_UNFOLD_BLOCKS; ++q)
        if (q < nq) Sb[q * N] = make_float2(ar[q], -ai[q]);
}

// position p < P of block blockIdx.y is handle output (j0 + b) P - off0 + p, at span position N - P + p; outputs below
// n_lo (before the handle's output 0, or before this call's first) are not stored, output n lands at out[n - n_lo]
__global__ void __launch_bounds__(256) fcsb_store_kernel(const float2 *__restrict__ X, long long N, long long P,
                                                         long long off0, long long j0, long long n_lo, float inv_n,
                                                         float2 *__restrict__ out) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const long long b = blockIdx.y;
    const long long n = (j0 + b) * P - off0 + p;
    if (n < n_lo) return;
    const float2 v = X[b * N + N - P + p];
    out[n - n_lo] = make_float2(v.x * inv_n, -v.y * inv_n);
}

// copies channel blockIdx.y's frames [lo_k, end_k) (from lq Il / I_k, the new carried frames) into row k of dst
__global__ void __launch_bounds__(256) fcsb_carry_kernel(FcsbSrc src, const FcsbChan *__restrict__ chan, long long lq,
                                                         long long eq, long long hs, float2 *__restrict__ dst) {
    const int k = blockIdx.y;
    const long long fil = chan[k].fil, lo = lq * fil, cnt = (eq - lq) * fil;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < cnt; t += (long long)gridDim.x * blockDim.x)
        dst[k * hs + t] = fcsb_load(src, k, fil, lo + t);
}

}  // namespace

struct FcsbHost {
    int dev = 0;
    size_t L = 0, C = 0, n_sets = 1;
    uint64_t first = 0;
    std::vector<float> taps;         // n_sets x L, as given
    std::vector<uint64_t> inc;
    std::vector<size_t> I;
    long long N = 0, P = 0, Il = 1, Imin = 1, off0 = 0;  // off0: handle block 0 starts at handle output -off0
    long long rows = 0;              // sum over channels of M_k (c64 per block in the gather / small-transform buffers)
    std::vector<FcsbChan> chan;
    std::vector<std::pair<long long, long long>> groups;  // (M, first channel of the group in `order`)
    std::vector<int> order;          // channels sorted by group
    long long total = 0;             // output positions seen (a multiple of Il)
    long long hist_lo = 0;           // d_hist[cur] row k holds channel k's frames from hist_lo / I_k to total / I_k
    long long hist_stride = 0;       // c64 per row of d_hist[cur]
};

using FftPlan = Owned<sdr_fft_t, sdr_fft_destroy>;

struct sdr_fcsb : FcsbHost {
    StreamRef stream;
    FftPlan big;                     // the N-point plan
    std::vector<FftPlan> small;      // one per group
    DevBuf d_G, d_tab, d_chan, d_mb;
    DevBuf d_hist[2];
    int cur = 0;
    DevBuf d_v, d_V, d_S, d_X, d_in, d_out;

    int alloc(void *user_stream, const sdr_fcsb *src);
    int copy_device(const sdr_fcsb &src);
};

// host-side geometry of a handle whose configuration fields are set: N, P, per-channel constants, groups
static int fcsb_geometry_fields(FcsbHost *h) {
    size_t n = 0, p = 0;
    int rc = sdr_fcfb_geometry(h->L, h->I.data(), h->C, &n, &p);
    if (rc) return rc;
    h->N = (long long)n;
    h->P = (long long)p;
    h->Il = 1;
    for (size_t I : h->I) h->Il = h->Il / (long long)gcd_u((unsigned long long)h->Il, I) * (long long)I;
    h->Imin = (long long)*std::min_element(h->I.begin(), h->I.end());
    const uint64_t eps = h->first % (uint64_t)h->Il;
    h->off0 = (long long)((h->first - eps) % (uint64_t)h->P);
    h->chan.assign(h->C, FcsbChan{});
    for (size_t k = 0; k < h->C; ++k) {
        FcsbChan &c = h->chan[k];
        c.I = (long long)h->I[k];
        const long long g = c.I & -c.I;
        c.M = h->N / g;
        c.us = c.I / g;
        c.rho = fcfb_rho(h->N, h->P, c.I);
        c.nfr = (h->N - c.rho + c.I - 1) / c.I;
        c.fpb = h->P / c.I;
        // span frame 0 of block j sits at handle output (j + 1) P - off0 - N + rho, a frame position (exact division)
        c.fr0 = (c.rho + 1 - h->N - h->off0) / c.I - 1;
        c.fil = h->Il / c.I;
        c.inc = h->inc[k];
    }
    // groups of equal M, largest first; rows of a group are (channel, block) in slab order
    h->order.resize(h->C);
    for (size_t k = 0; k < h->C; ++k) h->order[k] = (int)k;
    std::stable_sort(h->order.begin(), h->order.end(), [&](int a, int b) { return h->chan[a].M > h->chan[b].M; });
    h->groups.clear();
    long long base = 0;
    for (size_t i = 0; i < h->C; ++i) {
        FcsbChan &c = h->chan[h->order[i]];
        if (h->groups.empty() || h->groups.back().first != c.M) h->groups.push_back({c.M, (long long)i});
        c.base = base;
        base += c.M;
    }
    h->rows = base;
    return SDR_OK;
}

// G'_k (C rows of N, the conjugate rho factor of K9's) and the rotation tables tab[k][r] = e^{+2 pi i r I_k Delta_k}
// (C rows of FCSB_RUN), f64 on the host, rounded to f32 once
static void fcsb_tables(const FcsbHost *h, std::vector<float2> &G, std::vector<float2> &tab) {
    const long long N = h->N, L = (long long)h->L;
    G.assign((size_t)h->C * N, make_float2(0.f, 0.f));
    tab.assign((size_t)h->C * FCSB_RUN, make_float2(0.f, 0.f));
    for (size_t k = 0; k < h->C; ++k) {
        const FcsbChan &c = h->chan[k];
        const float *hk = h->taps.data() + (h->n_sets == 1 ? 0 : k * h->L);
        fc_spectrum(hk, L, c.inc, N, c.rho, -1, G.data() + (size_t)k * N);
        for (int r = 0; r < FCSB_RUN; ++r) {
            const double t = NCO_2PI * nco_turns((uint64_t)c.I * (uint64_t)r * c.inc);
            tab[(size_t)k * FCSB_RUN + r] = make_float2((float)std::cos(t), (float)std::sin(t));
        }
    }
}

static int fcsb_plan(const sdr_fcsb *h, long long n, FftPlan &out) {
    sdr_fft_config_t fc;
    fc.n = (size_t)n;
    fc.input_format = SDR_FMT_C64;
    fc.flags = 0;
    fc.device = h->dev;
    fc.stream = (void *)h->stream.s;
    int rc = SDR_OK;
    out.reset(sdr_fft_create(&fc, &rc));
    return out ? SDR_OK : rc;
}

// plans, tables and history buffers of a handle whose geometry fields are set; src != null copies src's tables
inline int sdr_fcsb::alloc(void *user_stream, const sdr_fcsb *src) {
    int rc = stream.init(user_stream);
    if (rc) return rc;
    cudaStream_t st = stream.s;
    if ((rc = fcsb_plan(this, N, big))) return rc;
    small.resize(groups.size());
    for (size_t q = 0; q < groups.size(); ++q)
        if ((rc = fcsb_plan(this, groups[q].first, small[q]))) return rc;
    const size_t gbytes = C * (size_t)N * sizeof(float2), tbytes = C * FCSB_RUN * sizeof(float2);
    if (src) {
        if ((rc = d_G.alloc(gbytes)) || (rc = d_tab.alloc(tbytes))) return rc;
        SDR_CUDA_TRY(cudaMemcpyAsync(d_G.p, src->d_G.p, gbytes, cudaMemcpyDeviceToDevice, st));
        SDR_CUDA_TRY(cudaMemcpyAsync(d_tab.p, src->d_tab.p, tbytes, cudaMemcpyDeviceToDevice, st));
    } else {
        std::vector<float2> G, tab;
        fcsb_tables(this, G, tab);
        if ((rc = d_G.upload(G.data(), gbytes, st)) || (rc = d_tab.upload(tab.data(), tbytes, st))) return rc;
        SDR_CUDA_TRY(cudaStreamSynchronize(st));  // the host vectors go out of scope
    }
    std::vector<longlong2> mb(C);
    for (size_t k = 0; k < C; ++k) mb[k] = make_longlong2(chan[k].M, chan[k].base);
    if ((rc = d_chan.upload(chan.data(), C * sizeof(FcsbChan), st))) return rc;
    if ((rc = d_mb.upload(mb.data(), C * sizeof(longlong2), st))) return rc;
    for (int i = 0; i < 2; ++i)
        if ((rc = d_hist[i].reserve(16))) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

// the carried frames
inline int sdr_fcsb::copy_device(const sdr_fcsb &src) {
    const size_t bytes = C * (size_t)hist_stride * sizeof(float2);
    if (bytes == 0) return SDR_OK;
    int rc = d_hist[0].reserve(bytes);
    if (rc) return rc;
    return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, bytes, cudaMemcpyDeviceToDevice));
}

extern "C" sdr_fcsb_t *sdr_fcsb_create(const sdr_fcsb_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || !cfg->phase_inc || !cfg->interpolation || cfg->n_taps == 0 ||
        cfg->n_taps > FCSB_MAX_TAPS || cfg->n_channels == 0 || cfg->n_channels > FCSB_MAX_CH ||
        (cfg->n_tap_sets != 1 && cfg->n_tap_sets != cfg->n_channels))
        return fail(err, SDR_ERR_INVALID_ARG);
    for (size_t k = 0; k < cfg->n_channels; ++k)
        if (cfg->interpolation[k] == 0) return fail(err, SDR_ERR_INVALID_ARG);
    for (size_t i = 0; i < cfg->n_taps * cfg->n_tap_sets; ++i)
        if (!std::isfinite(cfg->taps[i])) return fail(err, SDR_ERR_INVALID_ARG);
    size_t n_fft = 0, hop = 0;
    const int rc = sdr_fcfb_geometry(cfg->n_taps, cfg->interpolation, cfg->n_channels, &n_fft, &hop);
    if (rc) return fail(err, rc);
    return create_handle<sdr_fcsb>(err, cfg->device, cfg->stream, [&](sdr_fcsb &h) {
        h.L = cfg->n_taps;
        h.C = cfg->n_channels;
        h.n_sets = cfg->n_tap_sets;
        h.first = cfg->first_sample;
        h.taps.assign(cfg->taps, cfg->taps + h.L * h.n_sets);
        h.inc.assign(cfg->phase_inc, cfg->phase_inc + h.C);
        h.I.assign(cfg->interpolation, cfg->interpolation + h.C);
        return fcsb_geometry_fields(&h);
    });
}

extern "C" void sdr_fcsb_destroy(sdr_fcsb_t *h) { destroy_handle(h); }

extern "C" int sdr_fcsb_reset(sdr_fcsb_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // frames below index 0 read as zero, so the stale carried frames are never used
    h->total = h->hist_lo = h->hist_stride = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_fcsb_t *sdr_fcsb_clone(const sdr_fcsb_t *src, int *err) { return clone_handle<FcsbHost>(src, err); }

// blocks completed by the first T output positions, and the outputs among them
static long long fcsb_blocks(const sdr_fcsb *h, long long T) { return (T + h->off0) / h->P; }
static long long fcsb_outputs(const sdr_fcsb *h, long long T) {
    return std::max(0LL, fcsb_blocks(h, T) * h->P - h->off0);
}

extern "C" size_t sdr_fcsb_output_count(const sdr_fcsb_t *h, size_t n_time) {
    if (!h || n_time > (size_t)(LLONG_MAX / 2 - h->total)) return 0;
    return (size_t)(fcsb_outputs(h, h->total + (long long)n_time) - fcsb_outputs(h, h->total));
}

// blocks jA .. jB - 1 through the five stages, in slabs; outputs from handle output n_lo on to out
static int fcsb_blocks_run(sdr_fcsb *h, const FcsbSrc &src, long long jA, long long jB, long long n_lo, float2 *out) {
    cudaStream_t st = h->stream.s;
    const long long N = h->N;
    const long long step = std::max<long long>(1, std::min<long long>({(long long)(FCSB_SLAB_BYTES / (8 * N)),
                                                                        (long long)(FCSB_ROWS_BYTES / (8 * h->rows)), 65535}));
    const long long B = std::min(step, jB - jA);
    int rc = h->d_v.reserve((size_t)(B * h->rows) * sizeof(float2));
    if (!rc) rc = h->d_V.reserve((size_t)(B * h->rows) * sizeof(float2));
    if (!rc) rc = h->d_S.reserve((size_t)(B * N) * sizeof(float2));
    if (!rc) rc = h->d_X.reserve((size_t)(B * N) * sizeof(float2));
    if (rc) return rc;
    long long max_m = 0;
    for (const FcsbChan &c : h->chan) max_m = std::max(max_m, c.M);
    const uint64_t first = h->first;
    const float inv_n = 1.0f / (float)N;  // exact: N is a power of two
    for (long long j0 = jA; j0 < jB; j0 += B) {
        const long long nb = std::min(B, jB - j0);
        dim3 gg((unsigned)((max_m + 255) / 256), (unsigned)h->C, (unsigned)nb);
        fcsb_gather_kernel<<<gg, 256, 0, st>>>(src, (const FcsbChan *)h->d_chan.p, (const float2 *)h->d_tab.p, N, nb,
                                               j0, first, (float2 *)h->d_v.p);
        count_launch();
        if ((rc = launch_status())) return rc;
        for (size_t q = 0; q < h->groups.size(); ++q) {
            const long long first_ch = h->groups[q].second;
            const long long last = q + 1 < h->groups.size() ? h->groups[q + 1].second : (long long)h->C;
            const size_t off = (size_t)(nb * h->chan[h->order[first_ch]].base);
            rc = sdr_fft_exec_dev(h->small[q].get(), (const float2 *)h->d_v.p + off, (size_t)((last - first_ch) * nb),
                                  (float *)((float2 *)h->d_V.p + off));
            if (rc) return rc;
        }
        dim3 gu((unsigned)((N + 255) / 256), (unsigned)((nb + FCSB_UNFOLD_BLOCKS - 1) / FCSB_UNFOLD_BLOCKS));
        fcsb_unfold_kernel<<<gu, 256, 0, st>>>((const float2 *)h->d_V.p, (const float2 *)h->d_G.p,
                                               (const longlong2 *)h->d_mb.p, (int)h->C, N, nb, (float2 *)h->d_S.p);
        count_launch();
        if ((rc = launch_status())) return rc;
        if ((rc = sdr_fft_exec_dev(h->big.get(), h->d_S.p, (size_t)nb, (float *)h->d_X.p))) return rc;
        dim3 gs((unsigned)((h->P + 255) / 256), (unsigned)nb);
        fcsb_store_kernel<<<gs, 256, 0, st>>>((const float2 *)h->d_X.p, N, h->P, h->off0, j0, n_lo, inv_n, out);
        count_launch();
        if ((rc = launch_status())) return rc;
    }
    return SDR_OK;
}

// in: C device rows of n_time / I_k frames, row stride in_stride; out: the outputs of the blocks this call completes
static int fcsb_run(sdr_fcsb *h, const float2 *in, long long n_time, long long in_stride, float2 *out) {
    cudaStream_t st = h->stream.s;
    const long long end = h->total + n_time;
    const long long jA = fcsb_blocks(h, h->total), jB = fcsb_blocks(h, end);
    FcsbSrc src;
    src.hist = (const float2 *)h->d_hist[h->cur].p;
    src.in = in;
    src.hs = h->hist_stride;
    src.is = in_stride;
    src.hq = h->hist_lo / h->Il;
    src.iq = h->total / h->Il;
    if (jB > jA) {
        const int rc = fcsb_blocks_run(h, src, jA, jB, fcsb_outputs(h, h->total), out);
        if (rc) return rc;
    }
    // carry the frames of block jB's span so far: from lo (rounded down to a multiple of Il) to end
    const long long span_lo = (jB + 1) * h->P - h->off0 - h->N;
    const long long lo = std::min(end, std::max(0LL, span_lo) / h->Il * h->Il);
    const long long hs = (end - lo) / h->Imin;
    if (hs > 0) {
        DevBuf &dst = h->d_hist[h->cur ^ 1];
        int rc = dst.reserve(h->C * (size_t)hs * sizeof(float2));
        if (rc) return rc;
        const unsigned gx = (unsigned)std::min<long long>((hs + 255) / 256, 1024);
        fcsb_carry_kernel<<<dim3(gx, (unsigned)h->C), 256, 0, st>>>(src, (const FcsbChan *)h->d_chan.p, lo / h->Il,
                                                                    end / h->Il, hs, (float2 *)dst.p);
        count_launch();
        if ((rc = launch_status())) return rc;
        h->cur ^= 1;
    }
    h->hist_lo = lo;
    h->hist_stride = hs;
    h->total = end;
    return SDR_OK;
}

static int fcsb_check(const sdr_fcsb *h, const float *in, size_t n_time, size_t in_stride, const float *out,
                      size_t out_cap, size_t *n_out, size_t *cnt) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    *n_out = 0;
    if (n_time % (size_t)h->Il != 0) return SDR_ERR_INVALID_ARG;
    // handle positions stay far inside int64
    if (n_time > (size_t)(LLONG_MAX / 2 - h->total)) return SDR_ERR_INVALID_ARG;
    if (n_time > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < n_time / (size_t)h->Imin) return SDR_ERR_INVALID_ARG;
    *cnt = sdr_fcsb_output_count(h, n_time);
    if (*cnt > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (*cnt > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    return SDR_OK;
}

extern "C" int sdr_fcsb_process_dev(sdr_fcsb_t *h, const float *in_c64, size_t n_time, size_t in_stride,
                                    float *out_c64, size_t out_cap, size_t *n_out) {
    size_t cnt = 0;
    int rc = fcsb_check(h, in_c64, n_time, in_stride, out_c64, out_cap, n_out, &cnt);
    if (rc || n_time == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const long long stride = h->C > 1 ? (long long)in_stride : (long long)(n_time / h->I[0]);
    rc = fcsb_run(h, (const float2 *)in_c64, (long long)n_time, stride, (float2 *)out_c64);
    if (rc) return rc;
    *n_out = cnt;
    return SDR_OK;
}

extern "C" int sdr_fcsb_process(sdr_fcsb_t *h, const float *in_c64, size_t n_time, size_t in_stride, float *out_c64,
                                size_t out_cap, size_t *n_out) {
    size_t cnt = 0;
    int rc = fcsb_check(h, in_c64, n_time, in_stride, out_c64, out_cap, n_out, &cnt);
    if (rc || n_time == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C, Il = (size_t)h->Il, Imin = (size_t)h->Imin;
    const size_t stride = C > 1 ? in_stride : n_time / h->I[0];
    cudaStream_t st = h->stream.s;
    // chunks of output positions (multiples of Il) with at most ~32 MiB of output and of input: H2D, compute, D2H in
    // stream order; runs of consecutive channels with equal I go up in one 2-D copy
    size_t chunk = std::min(FCSB_HOST_BYTES / 8, FCSB_HOST_BYTES / (8 * C) * Imin) / Il * Il;
    chunk = std::min(std::max(chunk, Il), n_time);
    const size_t cs = chunk / Imin;                  // device row stride of one chunk's frames
    const size_t ocap = chunk + (size_t)h->P;         // outputs one chunk can complete
    rc = h->d_in.reserve(C * cs * 8);
    if (!rc) rc = h->d_out.reserve(ocap * 8);
    if (rc) return rc;
    size_t done = 0, made = 0;
    while (done < n_time) {
        const size_t cn = std::min(chunk, n_time - done);
        const size_t part = sdr_fcsb_output_count(h, cn);
        for (size_t k0 = 0; k0 < C;) {
            size_t k1 = k0 + 1;
            while (k1 < C && h->I[k1] == h->I[k0]) ++k1;
            const size_t Ik = h->I[k0];
            SDR_CUDA_TRY(cudaMemcpy2DAsync((float2 *)h->d_in.p + k0 * cs, cs * 8, in_c64 + 2 * (k0 * stride + done / Ik),
                                           stride * 8, cn / Ik * 8, k1 - k0, cudaMemcpyHostToDevice, st));
            k0 = k1;
        }
        rc = fcsb_run(h, (const float2 *)h->d_in.p, (long long)cn, (long long)cs, (float2 *)h->d_out.p);
        if (rc) return rc;
        if (part > 0)
            SDR_CUDA_TRY(cudaMemcpyAsync(out_c64 + 2 * made, h->d_out.p, part * 8, cudaMemcpyDeviceToHost, st));
        made += part;
        done += cn;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_out = made;
    return SDR_OK;
}

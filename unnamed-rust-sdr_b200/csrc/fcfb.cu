// fcfb.cu -- K9, sdr_fcfb_*: fast-convolution (overlap-save) channel bank.  C channels of one IQ stream, each mixed to
// 0 Hz by its own 64-bit NCO, low-pass filtered by real taps h_k and decimated by its own D_k -- sdr_ddc's channel with
// a per-channel D -- computed in the rotated-taps form
//     y_k[m] = e^{-2 pi i phi_k(F + n_m) / 2^64} (g_k * x)[n_m],  g_k[j] = h_k[j] e^{+2 pi i (j Delta_k mod 2^64) / 2^64}
// by overlap-save on blocks of the absolute stream grid.
//
// Geometry (sdr_fcfb_geometry): Dl = lcm(D_k), N = the smallest power of two >= 1024 with P = floor((N - L + 1) / Dl) Dl
// >= N / 2.  Block b holds the outputs at absolute indices [b P + eps, (b + 1) P + eps), eps = F mod Dl; its span is the
// N inputs ending at (b + 1) P + eps - 1, so every channel's kept outputs sit at the same span positions
// t = N - P + D_k - 1 + i D_k, i < P / D_k, and N - P >= L - 1 makes the cyclic convolution exact there.
//
// Per slab of whole blocks (about 32 MiB of spectra, a few waves of the N-point plan):
//   fcfb_gather_kernel   span -> c64 (u8 unpacked, x[<0] = 0), read through (carried tail, caller block) pointers
//   sdr_fft plan N       X_b = DFT_N(span), once per block for all channels
//   fcfb_fold_kernel     F_kb[r] = sum_{a < g_k} G'_k[r + a M_k] X_b[r + a M_k],  M_k = N / g_k, g_k = the largest power
//                        of two dividing D_k, G'_k[r] = DFT_N(g_k)[r] e^{+2 pi i r rho_k / N}, rho_k = (N - P - 1) mod
//                        D_k (host f64, rounded to f32 once); writes conj(F) in rows grouped by M_k
//   sdr_fft plans M_k    one per distinct M_k: the inverse through conjugation, IDFT(F) = conj(DFT(conj F))
//   fcfb_store_kernel    (1/N) conj(.) is (g_k * x) at span position g_k u + rho_k; keeps u = u0_k + i D_k / g_k,
//                        derotates and stores channel-major rows at the caller's stride
// Derotation as K7: one f64 sincospi of the exact integer phase per (block, channel, run of 1024 outputs) times a
// per-channel f32 table of 1024 entries.  Every output depends only on its block's N samples and its absolute
// position, so blockings, addresses, clones and block-aligned shards give the same bits.
#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "nco.cuh"

using namespace sdr;

namespace {

constexpr size_t FCFB_MAX_CH = 256;
constexpr size_t FCFB_MAX_TAPS = (size_t)1 << 20;
constexpr long long FCFB_MIN_N = 1024;
constexpr long long FCFB_MAX_N = 1LL << 22;
constexpr size_t FCFB_SLAB_BYTES = (size_t)32 << 20;  // c64 spectra of one slab (a few waves of the N-point plan)
constexpr size_t FCFB_ROWS_BYTES = (size_t)128 << 20; // at most this much of fold rows per slab
constexpr size_t FCFB_HOST_BYTES = (size_t)32 << 20;  // host-memory calls: input and output chunk size
constexpr int FCFB_RUN = 1024;                        // outputs per derotation base (table length)
constexpr int FCFB_FOLD_BLOCKS = 4;                   // blocks per fold thread (G' read once for all of them)
constexpr int FCFB_STORE_BLOCKS = 64;                 // most blocks per store CTA (short runs)

struct FcfbChan {
    long long M;       // inverse size N / g
    long long g;       // folds
    long long D;
    long long base;    // fold / inverse rows of this channel start at slab offset B * base (units of c64)
    long long u0, us;  // kept output i is inverse bin u0 + i us
    long long keep;    // P / D
    uint64_t inc;
};

// Stream sample i of one call: 0 for i < 0, hist[i - hist_lo] below in_lo (the carried tail), in[i - in_lo] from in_lo on
struct FcfbSrc {
    const void *hist;
    const void *in;
    long long hist_lo, in_lo;
};

template <bool U8>
__device__ __forceinline__ float2 fcfb_load(const FcfbSrc &s, long long i) {
    if (i < 0) return make_float2(0.f, 0.f);
    const bool h = i < s.in_lo;
    const void *base = h ? s.hist : s.in;
    const long long k = h ? i - s.hist_lo : i - s.in_lo;
    if (U8) return unpack_iq_u16(__ldg(reinterpret_cast<const uint16_t *>(base) + k));
    return __ldg(reinterpret_cast<const float2 *>(base) + k);
}

// spans of blocks j0 .. j0 + nb - 1 side by side; block j's span starts at (j + 1) P - off0 - N (handle index)
template <bool U8>
__global__ void __launch_bounds__(256) fcfb_gather_kernel(FcfbSrc src, long long N, long long P, long long off0,
                                                          long long j0, long long nb, float2 *__restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N) return;
    for (long long b = blockIdx.y; b < nb; b += gridDim.y)
        out[b * N + t] = fcfb_load<U8>(src, (j0 + b + 1) * P - off0 - N + t);
}

// thread = (channel blockIdx.y, bin r < M, FCFB_FOLD_BLOCKS blocks): conj(sum_a G'[r + a M] X_b[r + a M]), a ascending
__global__ void __launch_bounds__(256) fcfb_fold_kernel(const float2 *__restrict__ X, const float2 *__restrict__ G,
                                                        const FcfbChan *__restrict__ chan, long long N, long long nb,
                                                        float2 *__restrict__ f) {
    const int k = blockIdx.y;
    const long long M = chan[k].M, g = chan[k].g;
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= M) return;
    const long long b0 = (long long)blockIdx.z * FCFB_FOLD_BLOCKS;
    const float2 *Gk = G + (size_t)k * N + r;
    const float2 *Xb = X + b0 * N + r;
    float ar[FCFB_FOLD_BLOCKS], ai[FCFB_FOLD_BLOCKS];
#pragma unroll
    for (int q = 0; q < FCFB_FOLD_BLOCKS; ++q) ar[q] = ai[q] = 0.f;
    const int nq = (int)min((long long)FCFB_FOLD_BLOCKS, nb - b0);
    for (long long a = 0; a < g; ++a) {
        const float2 w = __ldg(Gk + a * M);
#pragma unroll
        for (int q = 0; q < FCFB_FOLD_BLOCKS; ++q) {
            if (q < nq) {
                const float2 x = __ldg(Xb + q * N + a * M);
                ar[q] = __fmaf_rn(w.x, x.x, ar[q]);
                ar[q] = __fmaf_rn(-w.y, x.y, ar[q]);
                ai[q] = __fmaf_rn(w.x, x.y, ai[q]);
                ai[q] = __fmaf_rn(w.y, x.x, ai[q]);
            }
        }
    }
    float2 *fk = f + nb * chan[k].base + b0 * M + r;
#pragma unroll
    for (int q = 0; q < FCFB_FOLD_BLOCKS; ++q)
        if (q < nq) fk[q * M] = make_float2(ar[q], -ai[q]);
}

// Channel blockIdx.y; outputs i of block j (of this slab's nb) in runs of rl = min(keep, FCFB_RUN), one derotation
// base per (block, run).  A CTA takes one run of up to FCFB_STORE_BLOCKS consecutive blocks (br = FCFB_RUN / rl of
// them when a block is one short run, so every CTA has about FCFB_RUN outputs): derotate (1/N) conj(y) and store.
// Block j's first output of channel k is handle output (j P - off0) / D_k; outputs below m_lo[k] (before the handle's
// first sample) are not stored, output m lands at out[k * out_stride + m - m_lo[k]].
__global__ void __launch_bounds__(256) fcfb_store_kernel(const float2 *__restrict__ y, const FcfbChan *__restrict__ chan,
                                                         const float2 *__restrict__ tab, long long nb, long long j0,
                                                         long long P, long long off0, uint64_t a0, float inv_n,
                                                         const long long *__restrict__ m_lo, float2 *__restrict__ out,
                                                         long long out_stride) {
    __shared__ float2 base_s[FCFB_STORE_BLOCKS];
    const int k = blockIdx.y;
    const FcfbChan c = chan[k];
    const long long rl = min(c.keep, (long long)FCFB_RUN), runs = (c.keep + rl - 1) / rl;
    const long long br = runs > 1 ? 1 : min((long long)FCFB_STORE_BLOCKS, FCFB_RUN / rl);
    const long long unit = blockIdx.x, run = unit % runs, zb = unit / runs * br;
    if (zb >= nb) return;
    const long long nbb = min(br, nb - zb), i0 = run * rl;
    // absolute index of block j's first sample = a0 + j P; output i0 + r of block j: a0 + j P + D - 1 + (i0 + r) D
    if (threadIdx.x < nbb)
        base_s[threadIdx.x] = nco_rot((a0 + (uint64_t)((j0 + zb + threadIdx.x) * P) + (uint64_t)(i0 * c.D)) * c.inc);
    __syncthreads();
    const long long mlo = m_lo[k];
    float2 *ok = out + (long long)k * out_stride - mlo;
    for (long long t = threadIdx.x; t < nbb * rl; t += blockDim.x) {
        const long long bb = t / rl, r = t - bb * rl, i = i0 + r;
        if (i >= c.keep) continue;
        const long long z = zb + bb;
        const long long m = ((j0 + z) * P - off0) / c.D + i;
        if (m < mlo) continue;
        const float2 v = y[nb * c.base + z * c.M + c.u0 + i * c.us];
        const float2 w = make_float2(v.x * inv_n, -v.y * inv_n);
        ok[m] = cmul(cmul(base_s[bb], __ldg(tab + (size_t)k * FCFB_RUN + r)), w);
    }
}

}  // namespace

extern "C" int sdr_fcfb_geometry(size_t n_taps, const size_t *decimation, size_t n_channels, size_t *n_fft, size_t *hop) {
    if (!decimation || !n_fft || !hop || n_taps == 0 || n_taps > FCFB_MAX_TAPS || n_channels == 0 ||
        n_channels > FCFB_MAX_CH)
        return SDR_ERR_INVALID_ARG;
    unsigned long long Dl = 1;
    for (size_t k = 0; k < n_channels; ++k) {
        const unsigned long long D = decimation[k];
        if (D == 0) return SDR_ERR_INVALID_ARG;
        if (D > (unsigned long long)FCFB_MAX_N) return SDR_ERR_UNSUPPORTED;
        Dl = Dl / gcd_u(Dl, D) * D;  // both <= 2^22 here: no overflow
        if (Dl > (unsigned long long)FCFB_MAX_N) return SDR_ERR_UNSUPPORTED;
    }
    for (long long N = FCFB_MIN_N; N <= FCFB_MAX_N; N <<= 1) {
        const long long span = N - (long long)n_taps + 1;
        if (span <= 0) continue;
        const long long P = span / (long long)Dl * (long long)Dl;
        if (P > 0 && 2 * P >= N) {
            *n_fft = (size_t)N;
            *hop = (size_t)P;
            return SDR_OK;
        }
    }
    return SDR_ERR_UNSUPPORTED;
}

struct FcfbHost {
    int dev = 0;
    size_t L = 0, C = 0, n_sets = 1;
    uint64_t first = 0;
    int fmt = SDR_FMT_U8IQ;
    std::vector<float> taps;         // n_sets x L, as given
    std::vector<uint64_t> inc;
    std::vector<size_t> D;
    long long N = 0, P = 0, Dl = 1, off0 = 0;  // off0: handle block 0 starts at handle index -off0
    long long rows = 0;              // sum over channels of M_k (c64 per block in the fold / inverse buffers)
    std::vector<FcfbChan> chan;
    std::vector<std::pair<long long, long long>> groups;  // (M, first channel of the group in `order`)
    std::vector<int> order;          // channels sorted by group
    long long total = 0;             // input samples seen
    long long hist_lo = 0;           // d_hist[cur] holds handle samples hist_lo .. total - 1
};

using FftPlan = Owned<sdr_fft_t, sdr_fft_destroy>;

struct sdr_fcfb : FcfbHost {
    StreamRef stream;
    FftPlan fwd;
    std::vector<FftPlan> inv;        // one per group
    DevBuf d_G, d_tab, d_chan, d_mlo;
    DevBuf d_hist[2];
    int cur = 0;
    DevBuf d_x, d_X, d_f, d_y, d_in, d_out;

    int alloc(void *user_stream, const sdr_fcfb *src);
    int copy_device(const sdr_fcfb &src);
};

static size_t fcfb_es(const FcfbHost *h) { return h->fmt == SDR_FMT_U8IQ ? 2 : 8; }

// host-side geometry of a handle whose configuration fields are set: N, P, per-channel fold constants, groups
static int fcfb_geometry_fields(FcfbHost *h) {
    size_t n = 0, p = 0;
    int rc = sdr_fcfb_geometry(h->L, h->D.data(), h->C, &n, &p);
    if (rc) return rc;
    h->N = (long long)n;
    h->P = (long long)p;
    h->Dl = 1;
    for (size_t D : h->D) h->Dl = h->Dl / (long long)gcd_u((unsigned long long)h->Dl, D) * (long long)D;
    const uint64_t eps = h->first % (uint64_t)h->Dl;
    h->off0 = (long long)((h->first - eps) % (uint64_t)h->P);
    h->chan.assign(h->C, FcfbChan{});
    for (size_t k = 0; k < h->C; ++k) {
        FcfbChan &c = h->chan[k];
        c.D = (long long)h->D[k];
        c.g = c.D & -c.D;
        c.M = h->N / c.g;
        const long long rho = fcfb_rho(h->N, h->P, c.D);
        c.u0 = (h->N - h->P + c.D - 1 - rho) / c.g;
        c.us = c.D / c.g;
        c.keep = h->P / c.D;
        c.inc = h->inc[k];
    }
    // groups of equal M, largest first; rows of a group are (channel, block) in slab order
    h->order.resize(h->C);
    for (size_t k = 0; k < h->C; ++k) h->order[k] = (int)k;
    std::stable_sort(h->order.begin(), h->order.end(), [&](int a, int b) { return h->chan[a].M > h->chan[b].M; });
    h->groups.clear();
    long long base = 0;
    for (size_t i = 0; i < h->C; ++i) {
        FcfbChan &c = h->chan[h->order[i]];
        if (h->groups.empty() || h->groups.back().first != c.M) h->groups.push_back({c.M, (long long)i});
        c.base = base;
        base += c.M;
    }
    h->rows = base;
    return SDR_OK;
}

// G'_k (C rows of N) and the derotation tables (C rows of FCFB_RUN), f64 on the host, rounded to f32 once
static void fcfb_tables(const FcfbHost *h, std::vector<float2> &G, std::vector<float2> &tab) {
    const long long N = h->N, L = (long long)h->L;
    G.assign((size_t)h->C * N, make_float2(0.f, 0.f));
    tab.assign((size_t)h->C * FCFB_RUN, make_float2(0.f, 0.f));
    for (size_t k = 0; k < h->C; ++k) {
        const FcfbChan &c = h->chan[k];
        const float *hk = h->taps.data() + (h->n_sets == 1 ? 0 : k * h->L);
        fc_spectrum(hk, L, c.inc, N, fcfb_rho(N, h->P, c.D), +1, G.data() + (size_t)k * N);
        for (int r = 0; r < FCFB_RUN; ++r) {
            const double t = NCO_2PI * nco_turns(((uint64_t)c.D * (uint64_t)r + (uint64_t)c.D - 1) * c.inc);
            tab[(size_t)k * FCFB_RUN + r] = make_float2((float)std::cos(t), (float)-std::sin(t));
        }
    }
}

static int fcfb_plan(const sdr_fcfb *h, long long n, FftPlan &out) {
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
int sdr_fcfb::alloc(void *user_stream, const sdr_fcfb *src) {
    int rc = stream.init(user_stream);
    if (rc) return rc;
    cudaStream_t st = stream.s;
    if ((rc = fcfb_plan(this, N, fwd))) return rc;
    inv.resize(groups.size());
    for (size_t q = 0; q < groups.size(); ++q)
        if ((rc = fcfb_plan(this, groups[q].first, inv[q]))) return rc;
    const size_t gbytes = C * (size_t)N * sizeof(float2), tbytes = C * FCFB_RUN * sizeof(float2);
    if (src) {
        if ((rc = d_G.alloc(gbytes)) || (rc = d_tab.alloc(tbytes))) return rc;
        SDR_CUDA_TRY(cudaMemcpyAsync(d_G.p, src->d_G.p, gbytes, cudaMemcpyDeviceToDevice, st));
        SDR_CUDA_TRY(cudaMemcpyAsync(d_tab.p, src->d_tab.p, tbytes, cudaMemcpyDeviceToDevice, st));
    } else {
        std::vector<float2> G, tab;
        fcfb_tables(this, G, tab);
        if ((rc = d_G.upload(G.data(), gbytes, st)) || (rc = d_tab.upload(tab.data(), tbytes, st))) return rc;
        SDR_CUDA_TRY(cudaStreamSynchronize(st));  // the host vectors go out of scope
    }
    if ((rc = d_chan.upload(chan.data(), C * sizeof(FcfbChan), st))) return rc;
    if ((rc = d_mlo.reserve(C * sizeof(long long)))) return rc;
    for (int i = 0; i < 2; ++i)
        if ((rc = d_hist[i].reserve(16))) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

// the history tail
int sdr_fcfb::copy_device(const sdr_fcfb &src) {
    const size_t tail = (size_t)(total - hist_lo) * fcfb_es(this);
    if (tail == 0) return SDR_OK;
    int rc = d_hist[0].reserve(tail);
    if (rc) return rc;
    return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, tail, cudaMemcpyDeviceToDevice));
}

extern "C" sdr_fcfb_t *sdr_fcfb_create(const sdr_fcfb_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || !cfg->phase_inc || !cfg->decimation || cfg->n_taps == 0 || cfg->n_taps > FCFB_MAX_TAPS ||
        cfg->n_channels == 0 || cfg->n_channels > FCFB_MAX_CH ||
        (cfg->n_tap_sets != 1 && cfg->n_tap_sets != cfg->n_channels) ||
        (cfg->input_format != SDR_FMT_U8IQ && cfg->input_format != SDR_FMT_C64))
        return fail(err, SDR_ERR_INVALID_ARG);
    for (size_t k = 0; k < cfg->n_channels; ++k)
        if (cfg->decimation[k] == 0) return fail(err, SDR_ERR_INVALID_ARG);
    for (size_t i = 0; i < cfg->n_taps * cfg->n_tap_sets; ++i)
        if (!std::isfinite(cfg->taps[i])) return fail(err, SDR_ERR_INVALID_ARG);
    size_t n_fft = 0, hop = 0;
    const int rc = sdr_fcfb_geometry(cfg->n_taps, cfg->decimation, cfg->n_channels, &n_fft, &hop);
    if (rc) return fail(err, rc);
    return create_handle<sdr_fcfb>(err, cfg->device, cfg->stream, [&](sdr_fcfb &h) {
        h.L = cfg->n_taps;
        h.C = cfg->n_channels;
        h.n_sets = cfg->n_tap_sets;
        h.first = cfg->first_sample;
        h.fmt = cfg->input_format;
        h.taps.assign(cfg->taps, cfg->taps + h.L * h.n_sets);
        h.inc.assign(cfg->phase_inc, cfg->phase_inc + h.C);
        h.D.assign(cfg->decimation, cfg->decimation + h.C);
        return fcfb_geometry_fields(&h);
    });
}

extern "C" void sdr_fcfb_destroy(sdr_fcfb_t *h) { destroy_handle(h); }

extern "C" int sdr_fcfb_reset(sdr_fcfb_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // samples below index 0 read as zero, so the stale tail is never used
    h->total = h->hist_lo = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_fcfb_t *sdr_fcfb_clone(const sdr_fcfb_t *src, int *err) { return clone_handle<FcfbHost>(src, err); }

// blocks completed by the first T inputs, and channel k's outputs among them
static long long fcfb_blocks(const sdr_fcfb *h, long long T) { return (T + h->off0) / h->P; }
static long long fcfb_outputs(const sdr_fcfb *h, size_t k, long long T) {
    return std::max(0LL, fcfb_blocks(h, T) * h->P - h->off0) / (long long)h->D[k];
}

extern "C" int sdr_fcfb_output_count(const sdr_fcfb_t *h, size_t n_in, size_t *counts) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!counts) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k)
        counts[k] = (size_t)(fcfb_outputs(h, k, h->total + (long long)n_in) - fcfb_outputs(h, k, h->total));
    return SDR_OK;
}

// blocks jA .. jB - 1 through the five stages, in slabs; outputs to C rows of out_stride
static int fcfb_blocks_run(sdr_fcfb *h, const FcfbSrc &src, long long jA, long long jB, float2 *out,
                           long long out_stride) {
    cudaStream_t st = h->stream.s;
    const long long N = h->N;
    const long long step = std::max<long long>(1, std::min<long long>({(long long)(FCFB_SLAB_BYTES / (8 * N)),
                                                                        (long long)(FCFB_ROWS_BYTES / (8 * h->rows)), 65535}));
    const long long B = std::min(step, jB - jA);
    int rc = h->d_x.reserve((size_t)(B * N) * sizeof(float2));
    if (!rc) rc = h->d_X.reserve((size_t)(B * N) * sizeof(float2));
    if (!rc) rc = h->d_f.reserve((size_t)(B * h->rows) * sizeof(float2));
    if (!rc) rc = h->d_y.reserve((size_t)(B * h->rows) * sizeof(float2));
    if (rc) return rc;
    std::vector<long long> mlo(h->C);
    for (size_t k = 0; k < h->C; ++k) mlo[k] = fcfb_outputs(h, k, h->total);
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_mlo.p, mlo.data(), h->C * sizeof(long long), cudaMemcpyHostToDevice, st));
    long long max_m = 0;
    for (const FcfbChan &c : h->chan) max_m = std::max(max_m, c.M);
    const uint64_t a0 = h->first - (uint64_t)h->off0;
    const float inv_n = 1.0f / (float)N;  // exact: N is a power of two
    for (long long j0 = jA; j0 < jB; j0 += B) {
        const long long nb = std::min(B, jB - j0);
        dim3 gg((unsigned)((N + 255) / 256), (unsigned)std::min<long long>(nb, 65535));
        if (h->fmt == SDR_FMT_U8IQ)
            fcfb_gather_kernel<true><<<gg, 256, 0, st>>>(src, N, h->P, h->off0, j0, nb, (float2 *)h->d_x.p);
        else
            fcfb_gather_kernel<false><<<gg, 256, 0, st>>>(src, N, h->P, h->off0, j0, nb, (float2 *)h->d_x.p);
        count_launch();
        if ((rc = launch_status())) return rc;
        if ((rc = sdr_fft_exec_dev(h->fwd.get(), h->d_x.p, (size_t)nb, (float *)h->d_X.p))) return rc;
        dim3 gf((unsigned)((max_m + 255) / 256), (unsigned)h->C, (unsigned)((nb + FCFB_FOLD_BLOCKS - 1) / FCFB_FOLD_BLOCKS));
        fcfb_fold_kernel<<<gf, 256, 0, st>>>((const float2 *)h->d_X.p, (const float2 *)h->d_G.p,
                                             (const FcfbChan *)h->d_chan.p, N, nb, (float2 *)h->d_f.p);
        count_launch();
        if ((rc = launch_status())) return rc;
        for (size_t q = 0; q < h->groups.size(); ++q) {
            const long long first = h->groups[q].second;
            const long long last = q + 1 < h->groups.size() ? h->groups[q + 1].second : (long long)h->C;
            const size_t off = (size_t)(nb * h->chan[h->order[first]].base);
            rc = sdr_fft_exec_dev(h->inv[q].get(), (const float2 *)h->d_f.p + off, (size_t)((last - first) * nb),
                                  (float *)((float2 *)h->d_y.p + off));
            if (rc) return rc;
        }
        long long units = 0;  // store CTAs of the channel that needs most (fcfb_store_kernel's split)
        for (const FcfbChan &c : h->chan) {
            const long long rl = std::min<long long>(c.keep, FCFB_RUN), runs = (c.keep + rl - 1) / rl;
            const long long br = runs > 1 ? 1 : std::min<long long>(FCFB_STORE_BLOCKS, FCFB_RUN / rl);
            units = std::max(units, (nb + br - 1) / br * runs);
        }
        dim3 gs((unsigned)units, (unsigned)h->C);
        fcfb_store_kernel<<<gs, 256, 0, st>>>((const float2 *)h->d_y.p, (const FcfbChan *)h->d_chan.p,
                                              (const float2 *)h->d_tab.p, nb, j0, h->P, h->off0, a0, inv_n,
                                              (const long long *)h->d_mlo.p, out, out_stride);
        count_launch();
        if ((rc = launch_status())) return rc;
    }
    return SDR_OK;
}

// in: n_in device samples; out: C rows of out_stride c64, the outputs of the blocks this call completes
static int fcfb_run(sdr_fcfb *h, const void *in, size_t n_in, float *out, size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t es = fcfb_es(h);
    const long long end = h->total + (long long)n_in;
    const long long jA = fcfb_blocks(h, h->total), jB = fcfb_blocks(h, end);
    FcfbSrc src;
    src.hist = h->d_hist[h->cur].p;
    src.in = in;
    src.hist_lo = h->hist_lo;
    src.in_lo = h->total;
    if (jB > jA) {
        const int rc = fcfb_blocks_run(h, src, jA, jB, (float2 *)out, (long long)out_stride);
        if (rc) return rc;
    }
    // carry the span of block jB so far: handle samples lo .. end - 1 (fewer than N)
    const long long lo = std::min(end, std::max(0LL, (jB + 1) * h->P - h->off0 - h->N));
    if (end > lo) {
        DevBuf &dst = h->d_hist[h->cur ^ 1];
        int rc = dst.reserve((size_t)(end - lo) * es);
        if (rc) return rc;
        const long long from_old = std::max(0LL, h->total - lo);
        if (from_old > 0)
            SDR_CUDA_TRY(cudaMemcpyAsync(dst.p, (const char *)src.hist + (size_t)(lo - h->hist_lo) * es,
                                         (size_t)from_old * es, cudaMemcpyDeviceToDevice, st));
        const long long first_in = std::max(lo, h->total);
        if (end > first_in)
            SDR_CUDA_TRY(cudaMemcpyAsync((char *)dst.p + (size_t)from_old * es,
                                         (const char *)in + (size_t)(first_in - h->total) * es,
                                         (size_t)(end - first_in) * es, cudaMemcpyDeviceToDevice, st));
        h->cur ^= 1;
    }
    h->hist_lo = lo;
    h->total = end;
    return SDR_OK;
}

static int fcfb_check(const sdr_fcfb *h, const void *in, size_t n_in, const float *out, size_t out_cap,
                      size_t out_stride, size_t *n_out, std::vector<size_t> &cnt) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = 0;
    if (n_in > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    cnt.resize(h->C);
    sdr_fcfb_output_count(h, n_in, cnt.data());
    const size_t most = *std::max_element(cnt.begin(), cnt.end());
    if (most > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (most > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (most > 0 && out_stride < most) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_fcfb_process_dev(sdr_fcfb_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                                    size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    int rc = fcfb_check(h, in, n_in, out_c64, out_cap, out_stride, n_out, cnt);
    if (rc) return rc;
    if (((uintptr_t)in % fcfb_es(h)) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = fcfb_run(h, in, n_in, out_c64, out_stride);
    if (rc) return rc;
    for (size_t k = 0; k < h->C; ++k) n_out[k] = cnt[k];
    return SDR_OK;
}

extern "C" int sdr_fcfb_process(sdr_fcfb_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                                size_t out_stride, size_t *n_out) {
    std::vector<size_t> cnt;
    int rc = fcfb_check(h, in, n_in, out_c64, out_cap, out_stride, n_out, cnt);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t es = fcfb_es(h), C = h->C;
    const size_t dmin = *std::min_element(h->D.begin(), h->D.end());
    cudaStream_t st = h->stream.s;
    // chunks of at most ~32 MiB of input and of output: H2D, compute, D2H in stream order
    size_t chunk = std::max<size_t>(1, FCFB_HOST_BYTES / es);
    chunk = std::max<size_t>(1, std::min(chunk, (FCFB_HOST_BYTES / (8 * C) + 1) * dmin));
    chunk = std::min(chunk, std::max<size_t>(n_in, 1));
    const size_t fcap = (chunk + (size_t)h->P) / dmin + 1;  // outputs one chunk can complete, per channel
    rc = h->d_in.reserve(chunk * es);
    if (!rc) rc = h->d_out.reserve(fcap * C * 8);
    if (rc) return rc;
    std::vector<size_t> done(C, 0), part(C);
    size_t done_in = 0;
    while (done_in < n_in) {
        const size_t cn = std::min(chunk, n_in - done_in);
        sdr_fcfb_output_count(h, cn, part.data());
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_in.p, (const char *)in + done_in * es, cn * es, cudaMemcpyHostToDevice, st));
        rc = fcfb_run(h, h->d_in.p, cn, (float *)h->d_out.p, fcap);
        if (rc) return rc;
        for (size_t k = 0; k < C; ++k) {
            if (part[k] > 0)
                SDR_CUDA_TRY(cudaMemcpyAsync(out_c64 + 2 * (k * out_stride + done[k]), (const float2 *)h->d_out.p + k * fcap,
                                             part[k] * 8, cudaMemcpyDeviceToHost, st));
            done[k] += part[k];
        }
        done_in += cn;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    for (size_t k = 0; k < C; ++k) n_out[k] = done[k];
    return SDR_OK;
}

// eq.cu -- K17, sdr_eq_*: adaptive equalizer bank.  C independent c64 symbol streams, one sample per symbol; channel k
// has N complex weights w[0..N) (one N for the handle, 1 <= N <= 64), a delay line x_{s-j} (zeros before the stream), a
// symbol total s and an adaptation set {M, mu, a, err_max, S}.  For each symbol s (sdr_b200.h states it in full):
//     P_j = w[j] x_{s-j}   (four products and two sums, each rounded on its own)
//     p_l = P_l (+ P_{l+32} when N > 32 and l + 32 < N), 0 for N <= l < W;  W = 2^ceil(log2 min(N, 32))
//     y_s = the pairwise tree over p_0..p_{W-1}, o = W/2, ..., 1:  p_l <- fl(p_l + p_{l+o})
//     g   = CMA (s < S): fl(fl(|y|^2) - R) y;   DD (s >= S): y - D_M(y) at radius a
//     y or g not finite: e_s = 0 and w stays; else e_s = clamp(g), u = mu e_s, w[j] <- w[j] - u conj(x_{s-j})
// Every f32 operation is rounded on its own and the summation order is fixed, so a float32 restatement reproduces y, e
// and the taps bit for bit.  One symbol out per symbol in, so a call's counts are its inputs: nothing is copied back.
// The taps, the last N - 1 symbols and s of every channel live on the device between calls.
#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "ptx.cuh"

using namespace sdr;

namespace {

constexpr size_t EQ_MAX_CH = 65536;
constexpr size_t EQ_MAX_TAPS = 64;
constexpr int EQ_TILE = 32;                          // symbols per staged tile
constexpr int EQ_YS = EQ_TILE + 1;                   // row stride of the y and e tiles (a pad against bank conflicts)
constexpr size_t EQ_HOST_BYTES = (size_t)32 << 20;  // host-memory calls: chunk size of input

struct EqChan {                // per channel, fixed at create
    unsigned long long S;      // symbols s < S adapt by CMA, s >= S by DD
    float mu, emax, R;         // step, clamp of each component of e, CMA modulus fl(a a)
    float dp, dq;              // DD decision (+-dp, +-dq) or (+-dq, +-dp): M = 2 (a, 0); M = 4 (c, c); M = 8 (p, q)
    int order2;                // M = 2: always the first form, whatever |y.re| and |y.im| are
};

// lanes of a segment of W per channel (W = 2^ceil(log2 min(N, 32)))
inline int eq_lanes(size_t N) {
    int W = 1;
    while ((size_t)W < std::min<size_t>(N, 32)) W <<= 1;
    return W;
}

// shared memory of one CTA: x tiles [2][G][N + TILE] (N - 1 carried symbols, TILE staged, one pad), y and e tiles
// [2][G][TILE + 1] each, G = 32 / W channels
inline size_t eq_smem_bytes(size_t N, int W) {
    const size_t G = 32 / W;
    return 2 * (G * (N + EQ_TILE) + 2 * G * EQ_YS) * sizeof(float2);
}

// the largest of eq_smem_bytes over every tap count (N = 1: W = 1, 32 channels per CTA)
inline size_t eq_smem_max() {
    size_t m = 0;
    for (size_t N = 1; N <= EQ_MAX_TAPS; ++N) m = std::max(m, eq_smem_bytes(N, eq_lanes(N)));
    return m;
}

// A CTA of two warps owns G = 32 / W channels.
//   warp 0 steps the G recurrences, a segment of W lanes per channel: lane l keeps w[l] (and w[l + 32] when N > 32) in
//          registers, reads x_{s-l} (x_{s-l-32}) from the shared tile one symbol ahead, and the products meet in a
//          __shfl_xor_sync tree of width W, so every lane of the segment holds y_s, e_s and its own update.  At the end
//          of a tile the segment copies its last N - 1 symbols into the other buffer's carried part.
//   warp 1 stores the PREVIOUS tile's y and e in row segments (e only when asked for) and then cp.asyncs the NEXT
//          tile's [G channels x 32 symbols] into the other buffer, behind its carried symbols
// One barrier per tile.  A segment whose channel has fewer symbols runs the warp's loop with its writes and updates
// predicated off, so the shuffles always see the full warp.  in and out may be the same rows (in place): a tile's
// outputs are stored one tile after its inputs were read.
__global__ void __launch_bounds__(64) eq_kernel(const EqChan *__restrict__ chans, float2 *__restrict__ taps,
                                                float2 *__restrict__ hist, unsigned long long *__restrict__ sym,
                                                const long long *__restrict__ n_in, int C, int N, int W,
                                                const float2 *in, long long in_stride, float2 *out, float2 *err,
                                                long long out_stride) {
    extern __shared__ float2 eq_smem[];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int G = 32 / W, RS = N + EQ_TILE, H = N - 1;
    float2 *s_x = eq_smem;                   // [2][G][RS]: row[j] for j < H carried, row[H + i] symbol i of the tile
    float2 *s_y = s_x + 2 * G * RS;          // [2][G][EQ_YS]
    float2 *s_e = s_y + 2 * G * EQ_YS;       // [2][G][EQ_YS]
    const int ch0 = blockIdx.x * G;
    const int nrows = min(G, C - ch0);
    const long long nr = lane < nrows ? n_in[ch0 + lane] : 0;  // lane r holds row r's count
    long long nmax = nr;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
    const long long ntiles = (nmax + EQ_TILE - 1) / EQ_TILE;

    auto count = [&](int r, long long base) {
        const long long c = __shfl_sync(0xffffffffu, nr, r);
        return (int)max(0ll, min((long long)EQ_TILE, c - base));
    };
    auto issue = [&](long long tile, int buf) {
        const long long base = tile * EQ_TILE;
        for (int r = 0; r < nrows; ++r)
            if (lane < count(r, base))
                cp_async8(&s_x[(buf * G + r) * RS + H + lane], in + (long long)(ch0 + r) * in_stride + base + lane);
        cp_async_commit();
    };

    // warp 0: segment g = channel ch0 + g, lane q of it
    const int g = lane / W, q = lane & (W - 1);
    const bool live = role == 0 && g < nrows;
    const int ch = ch0 + g;
    const long long n = __shfl_sync(0xffffffffu, nr, min(g, 31));
    const bool has0 = q < N, has1 = q + 32 < N;
    EqChan c{};
    float2 w0 = make_float2(0.f, 0.f), w1 = make_float2(0.f, 0.f);
    unsigned long long s = 0;
    if (role == 1 && ntiles > 0) {
        issue(0, 0);
        cp_async_wait<0>();
    }
    if (live) {
        c = chans[ch];
        s = sym[ch];
        if (has0) w0 = taps[(long long)ch * N + q];
        if (has1) w1 = taps[(long long)ch * N + q + 32];
        for (int j = q; j < H; j += W) s_x[g * RS + j] = hist[(long long)ch * H + j];
    }
    __syncthreads();
    // iteration t: warp 0 steps tile t; warp 1 stores tile t - 1 and loads tile t + 1 (both in buffer (t + 1) & 1)
    for (long long tile = 0; tile <= ntiles; ++tile) {
        const int buf = (int)(tile & 1);
        if (role == 0) {
            if (tile < ntiles) {
                const long long base = tile * EQ_TILE;
                const int cnt = (int)max(0ll, min((long long)EQ_TILE, n - base));
                const int cmax = (int)min((long long)EQ_TILE, nmax - base);  // the same in every lane of the warp
                const float2 *row = &s_x[(buf * G + g) * RS + H];           // row[i - j] = x_{s-j} at symbol i
                float2 *py = &s_y[(buf * G + g) * EQ_YS], *pe = &s_e[(buf * G + g) * EQ_YS];
                float2 x0n = has0 ? row[-q] : make_float2(0.f, 0.f);
                float2 x1n = has1 ? row[-q - 32] : make_float2(0.f, 0.f);
                for (int i = 0; i < cmax; ++i) {
                    const float2 x0 = x0n, x1 = x1n;
                    // the next symbol's loads leave the dependent chain (the row has a pad element)
                    if (has0) x0n = row[i + 1 - q];
                    if (has1) x1n = row[i + 1 - q - 32];
                    float pr = 0.f, pi = 0.f;
                    if (has0) {
                        pr = __fsub_rn(__fmul_rn(w0.x, x0.x), __fmul_rn(w0.y, x0.y));
                        pi = __fadd_rn(__fmul_rn(w0.x, x0.y), __fmul_rn(w0.y, x0.x));
                    }
                    if (has1) {
                        pr = __fadd_rn(pr, __fsub_rn(__fmul_rn(w1.x, x1.x), __fmul_rn(w1.y, x1.y)));
                        pi = __fadd_rn(pi, __fadd_rn(__fmul_rn(w1.x, x1.y), __fmul_rn(w1.y, x1.x)));
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        if (o < W) {
                            pr = __fadd_rn(pr, __shfl_xor_sync(0xffffffffu, pr, o, W));
                            pi = __fadd_rn(pi, __shfl_xor_sync(0xffffffffu, pi, o, W));
                        }
                    }
                    const float yr = pr, yi = pi;
                    // CMA and DD side by side, then a select: channels of one warp in different phases or with
                    // different orders do not diverge
                    const float eps = __fsub_rn(__fadd_rn(__fmul_rn(yr, yr), __fmul_rn(yi, yi)), c.R);
                    const bool first = c.order2 || fabsf(yr) >= fabsf(yi);
                    const float da = first ? c.dp : c.dq, db = first ? c.dq : c.dp;
                    const float gdr = __fsub_rn(yr, yr >= 0.f ? da : -da), gdi = __fsub_rn(yi, yi >= 0.f ? db : -db);
                    const bool cma = s < c.S;
                    const float gr = cma ? __fmul_rn(eps, yr) : gdr, gi = cma ? __fmul_rn(eps, yi) : gdi;
                    // a non-finite y gives a non-finite g in both algorithms
                    const bool ok = isfinite(gr) && isfinite(gi);
                    const float er = ok ? fminf(fmaxf(gr, -c.emax), c.emax) : 0.f;
                    const float ei = ok ? fminf(fmaxf(gi, -c.emax), c.emax) : 0.f;
                    const bool active = i < cnt;
                    if (active && q == 0) {
                        py[i] = make_float2(yr, yi);
                        pe[i] = make_float2(er, ei);
                    }
                    if (active && ok) {
                        const float ur = __fmul_rn(c.mu, er), ui = __fmul_rn(c.mu, ei);
                        if (has0) {
                            w0.x = __fsub_rn(w0.x, __fadd_rn(__fmul_rn(ur, x0.x), __fmul_rn(ui, x0.y)));
                            w0.y = __fsub_rn(w0.y, __fsub_rn(__fmul_rn(ui, x0.x), __fmul_rn(ur, x0.y)));
                        }
                        if (has1) {
                            w1.x = __fsub_rn(w1.x, __fadd_rn(__fmul_rn(ur, x1.x), __fmul_rn(ui, x1.y)));
                            w1.y = __fsub_rn(w1.y, __fsub_rn(__fmul_rn(ui, x1.x), __fmul_rn(ur, x1.y)));
                        }
                    }
                    s += active ? 1 : 0;
                }
                // the last N - 1 symbols seen become the next tile's carried part
                if (g < nrows) {
                    float2 *nxt = &s_x[((buf ^ 1) * G + g) * RS];
                    for (int j = q; j < H; j += W) nxt[j] = row[cnt - H + j];
                }
            }
        } else {
            const int nb = buf ^ 1;
            if (tile > 0) {
                const long long base = (tile - 1) * EQ_TILE;
                for (int r = 0; r < nrows; ++r) {
                    if (lane < count(r, base)) {
                        const long long at = (long long)(ch0 + r) * out_stride + base + lane;
                        out[at] = s_y[(nb * G + r) * EQ_YS + lane];
                        if (err) err[at] = s_e[(nb * G + r) * EQ_YS + lane];
                    }
                }
            }
            if (tile + 1 < ntiles) {
                issue(tile + 1, nb);
                cp_async_wait<0>();
            }
        }
        __syncthreads();
    }
    if (live) {
        if (has0) taps[(long long)ch * N + q] = w0;
        if (has1) taps[(long long)ch * N + q + 32] = w1;
        const float2 *last = &s_x[((int)(ntiles & 1) * G + g) * RS];
        for (int j = q; j < H; j += W) hist[(long long)ch * H + j] = last[j];
        if (q == 0) sym[ch] = s;
    }
}

}  // namespace

struct EqHost {
    int dev = 0;
    size_t C = 0, N = 0;
    int W = 1;
    std::vector<EqChan> chans;
    std::vector<float2> init;  // the creation taps, C rows of N
    bool fresh = true;         // the device state is the creation state's once uploaded
};

struct sdr_eq : EqHost {
    StreamRef stream;
    DevBuf d_chans, d_taps, d_hist, d_sym, d_n;
    std::vector<long long> n_host;
    DevBuf d_in, d_out, d_err;

    size_t hist_bytes() const { return C * std::max<size_t>(N - 1, 1) * sizeof(float2); }
    int alloc(void *user_stream, const sdr_eq *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(EqChan), stream.s))) return rc;
        if ((rc = d_taps.alloc(C * N * sizeof(float2)))) return rc;
        if ((rc = d_hist.alloc(hist_bytes()))) return rc;
        if ((rc = d_sym.alloc(C * sizeof(unsigned long long)))) return rc;
        if ((rc = d_n.alloc(C * sizeof(long long)))) return rc;
        // the limit is one attribute of eq_kernel per device, shared by every handle: set to what the largest
        // footprint needs, it admits every handle's launch whatever order handles are created in, and setting the
        // same value from any number of handles and threads is idempotent
        SDR_CUDA_TRY(cudaFuncSetAttribute(eq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eq_smem_max()));
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_eq &src) {
        SDR_CUDA_TRY(cudaMemcpy(d_taps.p, src.d_taps.p, C * N * sizeof(float2), cudaMemcpyDeviceToDevice));
        SDR_CUDA_TRY(cudaMemcpy(d_hist.p, src.d_hist.p, hist_bytes(), cudaMemcpyDeviceToDevice));
        return cuda_status(cudaMemcpy(d_sym.p, src.d_sym.p, C * sizeof(unsigned long long), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_eq_t *sdr_eq_create(const sdr_eq_config_t *cfg, int *err) {
    bool ok = cfg && cfg->adapt && cfg->n_taps >= 1 && cfg->n_taps <= EQ_MAX_TAPS && cfg->n_channels >= 1 &&
              cfg->n_channels <= EQ_MAX_CH && (cfg->n_adapt == 1 || cfg->n_adapt == cfg->n_channels) &&
              (cfg->n_tap_sets <= 1 || cfg->n_tap_sets == cfg->n_channels) && (cfg->n_tap_sets == 0 || cfg->taps);
    for (size_t i = 0; ok && i < cfg->n_tap_sets * cfg->n_taps * 2; ++i) ok = std::isfinite(cfg->taps[i]);
    for (size_t k = 0; ok && k < cfg->n_adapt; ++k) {
        const sdr_eq_adapt_t &a = cfg->adapt[k];
        const float R = a.radius * a.radius;
        ok = (a.order == 2 || a.order == 4 || a.order == 8) && a.mu >= 0.f && std::isfinite(a.mu) &&
             a.radius > 0.f && std::isfinite(a.radius) && std::isfinite(R) && a.err_max > 0.f &&
             std::isfinite(a.err_max);
    }
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_eq>(err, cfg->device, cfg->stream, [&](sdr_eq &h) {
        const size_t C = cfg->n_channels, N = cfg->n_taps;
        h.C = C;
        h.N = N;
        h.W = eq_lanes(N);
        h.chans.resize(C);
        h.init.assign(C * N, make_float2(0.f, 0.f));
        for (size_t k = 0; k < C; ++k) {
            const sdr_eq_adapt_t &a = cfg->adapt[cfg->n_adapt == 1 ? 0 : k];
            const double r = a.radius;
            float dp = a.radius, dq = 0.f;  // M = 2
            if (a.order == 4) dp = dq = (float)(r / std::sqrt(2.0));
            if (a.order == 8) {  // cos(pi/8) and sin(pi/8) from square roots, which round correctly everywhere
                dp = (float)(r * (std::sqrt(2.0 + std::sqrt(2.0)) / 2.0));
                dq = (float)(r * (std::sqrt(2.0 - std::sqrt(2.0)) / 2.0));
            }
            h.chans[k] = EqChan{a.cma_symbols, a.mu, a.err_max, a.radius * a.radius, dp, dq, a.order == 2 ? 1 : 0};
            if (cfg->n_tap_sets == 0) {
                h.init[k * N + (N - 1) / 2] = make_float2(1.f, 0.f);
            } else {
                const float *t = cfg->taps + (cfg->n_tap_sets == 1 ? 0 : k) * N * 2;
                for (size_t j = 0; j < N; ++j) h.init[k * N + j] = make_float2(t[2 * j], t[2 * j + 1]);
            }
        }
        return SDR_OK;
    });
}

extern "C" void sdr_eq_destroy(sdr_eq_t *h) { destroy_handle(h); }

extern "C" int sdr_eq_reset(sdr_eq_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    h->fresh = true;  // the next call uploads the creation taps and zeroes the delay lines and s
    return SDR_OK;
}

extern "C" sdr_eq_t *sdr_eq_clone(const sdr_eq_t *src, int *err) { return clone_handle<EqHost>(src, err); }

extern "C" int sdr_eq_get_taps(sdr_eq_t *h, size_t channel, float *taps_c64) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!taps_c64) return SDR_ERR_BAD_DATA_PTR;
    if (channel >= h->C) return SDR_ERR_INVALID_ARG;
    const size_t N = h->N;
    if (h->fresh) {
        std::copy(h->init.begin() + channel * N, h->init.begin() + (channel + 1) * N, (float2 *)taps_c64);
        return SDR_OK;
    }
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    SDR_CUDA_TRY(cudaMemcpyAsync(taps_c64, (const float2 *)h->d_taps.p + channel * N, N * sizeof(float2),
                                 cudaMemcpyDeviceToHost, h->stream.s));
    return cuda_status(cudaStreamSynchronize(h->stream.s));
}

// in: C device rows (row stride in_stride), row k of n_in[k] symbols; outputs: C rows of out_stride.  Asynchronous.
static int eq_run(sdr_eq *h, const float2 *in, const size_t *n_in, size_t in_stride, float2 *out, float2 *err,
                  size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C, N = h->N;
    h->n_host.assign(n_in, n_in + C);
    if (h->fresh) {
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_taps.p, h->init.data(), C * N * sizeof(float2), cudaMemcpyHostToDevice, st));
        SDR_CUDA_TRY(cudaMemsetAsync(h->d_hist.p, 0, h->hist_bytes(), st));
        SDR_CUDA_TRY(cudaMemsetAsync(h->d_sym.p, 0, C * sizeof(unsigned long long), st));
        h->fresh = false;
    }
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_n.p, h->n_host.data(), C * sizeof(long long), cudaMemcpyHostToDevice, st));
    const int G = 32 / h->W;
    eq_kernel<<<(unsigned)((C + G - 1) / G), 64, eq_smem_bytes(N, h->W), st>>>(
        (const EqChan *)h->d_chans.p, (float2 *)h->d_taps.p, (float2 *)h->d_hist.p, (unsigned long long *)h->d_sym.p,
        (const long long *)h->d_n.p, (int)C, (int)N, h->W, in, C > 1 ? (long long)in_stride : 0, out, err,
        C > 1 ? (long long)out_stride : 0);
    count_launch();
    return launch_status();
}

static int eq_check(const sdr_eq *h, const float *in, const size_t *n_in, size_t in_stride, const float *out,
                    size_t out_stride, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in) return SDR_ERR_BAD_DATA_PTR;
    *longest = *std::max_element(n_in, n_in + h->C);
    if (*longest == 0) return SDR_OK;
    if (!in || !out) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && (in_stride < *longest || out_stride < *longest)) return SDR_ERR_INVALID_ARG;
    if ((const void *)in == (const void *)out && h->C > 1 && in_stride != out_stride) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_eq_process_dev(sdr_eq_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                  float *out_c64, float *err_c64, size_t out_stride) {
    size_t longest = 0;
    int rc = eq_check(h, in_c64, n_in, in_stride, out_c64, out_stride, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0 || ((uintptr_t)err_c64 % 8) != 0)
        return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    return eq_run(h, (const float2 *)in_c64, n_in, in_stride, (float2 *)out_c64, (float2 *)err_c64, out_stride);
}

extern "C" int sdr_eq_process(sdr_eq_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                              float *out_c64, float *err_c64, size_t out_stride) {
    size_t longest = 0;
    int rc = eq_check(h, in_c64, n_in, in_stride, out_c64, out_stride, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t istride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : longest;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` symbols per channel: H2D, compute, D2H
    const size_t chunk = std::min(longest, std::max<size_t>(1, EQ_HOST_BYTES / (C * 8)));
    const bool equal = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_out.reserve(chunk * C * 8);
    if (!rc && err_c64) rc = h->d_err.reserve(chunk * C * 8);
    if (rc) return rc;
    std::vector<size_t> take(C);
    // one array of C rows of c64 between the host rows (stride hs, at column `at`) and the device rows (chunk apart)
    auto move = [&](void *host, size_t hs, void *dev, size_t at, cudaMemcpyKind kind) -> int {
        const size_t bytes = 8;
        char *hp = (char *)host + at * bytes;
        if (equal)
            return cuda_status(kind == cudaMemcpyHostToDevice
                                   ? cudaMemcpy2DAsync(dev, chunk * bytes, hp, hs * bytes, take[0] * bytes, C, kind, st)
                                   : cudaMemcpy2DAsync(hp, hs * bytes, dev, chunk * bytes, take[0] * bytes, C, kind,
                                                       st));
        for (size_t k = 0; k < C; ++k)
            if (take[k]) {
                char *hk = hp + k * hs * bytes, *dk = (char *)dev + k * chunk * bytes;
                SDR_CUDA_TRY(kind == cudaMemcpyHostToDevice
                                 ? cudaMemcpyAsync(dk, hk, take[k] * bytes, kind, st)
                                 : cudaMemcpyAsync(hk, dk, take[k] * bytes, kind, st));
            }
        return SDR_OK;
    };
    for (size_t at = 0; at < longest; at += chunk) {
        for (size_t k = 0; k < C; ++k) take[k] = n_in[k] > at ? std::min(chunk, n_in[k] - at) : 0;
        if ((rc = move((void *)in_c64, istride, h->d_in.p, at, cudaMemcpyHostToDevice))) return rc;
        rc = eq_run(h, (const float2 *)h->d_in.p, take.data(), chunk, (float2 *)h->d_out.p,
                    err_c64 ? (float2 *)h->d_err.p : nullptr, chunk);
        if (rc) return rc;
        if ((rc = move(out_c64, ostride, h->d_out.p, at, cudaMemcpyDeviceToHost))) return rc;
        if (err_c64 && (rc = move(err_c64, ostride, h->d_err.p, at, cudaMemcpyDeviceToHost))) return rc;
    }
    return cuda_status(cudaStreamSynchronize(st));
}

// csync.cu -- K16, sdr_csync_*: carrier recovery bank.  C independent c64 symbol streams, one sample per symbol; channel
// k has a decision-directed Costas loop {M, kp, ki, err_max, max_freq}.  The phase phi is a uint64 in units of 2^-64
// turn (nco.cuh), the frequency nu an int64 in units of 2^-40 turn per symbol with |nu| <= V = floor(max_freq 2^40),
// q(x) = rint(x 2^40) for an f32 x.  From phi_0, nu_0, for s = 0, 1, ...:
//     r_s = nco_rot_fast(phi_s),  z_s = x_s r_s  (four products and two sums, each rounded on its own)
//     e_s = 0 for a non-finite g = D_M(z_s), else min(max(g, -err_max), err_max)
//     nu_{s+1} = clamp(nu_s + q(fl(ki e_s)), -V, V)
//     phi_{s+1} = phi_s + 2^24 (nu_{s+1} + q(fl(kp e_s)))   (mod 2^64)
// D_M is GNU Radio's order-M Costas detector with a = sgn(z.re) z.im, b = sgn(z.im) z.re (sgn(-0) = +1):
//     M = 2: a;  M = 4: fl(a - b);  M = 8: |z.re| >= |z.im| ? fl(a - fl(K b)) : fl(fl(K a) - b),  K = f32(sqrt 2 - 1)
// Every f32 operation of the product, the detector and the loop is rounded on its own (nothing is contracted), so a
// float32 restatement gives e_s from z_s bit for bit and integer arithmetic gives phi and nu from e_s.
// One symbol out per symbol in, so a call's counts are its inputs: nothing is copied back.  The loop keeps no history
// of symbols; phi and nu of every channel live on the device between calls.
#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "nco.cuh"
#include "ptx.cuh"

using namespace sdr;

namespace {

constexpr size_t CS_MAX_CH = 65536;
constexpr int CS_TILE = 32;                          // symbols per staged tile
constexpr size_t CS_HOST_BYTES = (size_t)32 << 20;  // host-memory calls: chunk size of input

struct CsChan {       // per channel, fixed at create
    float kp, ki, emax;
    float K;          // the M = 8 detector's f32(sqrt 2 - 1); 1 for M = 4, whose two branches are then both fl(a - b)
    long long V;      // bound of |nu|, 2^-40 turn per symbol
    int order2;       // M = 2: the detector is a alone
    int pad;
};

struct CsState {      // per channel, on the device between calls
    unsigned long long phi;
    long long nu;
};

// q(x) = rint(x 2^40) for an f32 x (|x| < 1/4: the scaling is exact and the result fits)
__device__ __forceinline__ long long cs_q(float x) { return __float2ll_rn(__fmul_rn(x, 0x1p40f)); }

// D_M(z): selects, not branches, so channels of one warp with different orders do not diverge
__device__ __forceinline__ float cs_detector(const CsChan &c, float zr, float zi) {
    const float a = zr >= 0.f ? zi : -zi, b = zi >= 0.f ? zr : -zr;
    const float g = fabsf(zr) >= fabsf(zi) ? __fsub_rn(a, __fmul_rn(c.K, b)) : __fsub_rn(__fmul_rn(c.K, a), b);
    return c.order2 ? a : g;
}

// A CTA of two warps owns 32 channels, one lane of each warp per channel (pll_kernel's layout).
//   warp 0 steps the 32 recurrences, nothing else: per symbol one shared load (prefetched) and three shared stores
//   warp 1 stores the PREVIOUS tile's z, phi and e in row segments (phi and e only when asked for) and then cp.asyncs
//          the NEXT tile's [32 channels x 32 symbols] into the same buffer in 256-byte row segments
// z replaces x in the tile it was computed from, so the output tile costs no shared memory of its own.  One barrier per
// tile.  A lane whose channel has fewer symbols idles.  in and out may be the same rows (in place): a tile's outputs
// are stored one tile after its inputs were read.
__global__ void __launch_bounds__(64) csync_kernel(const CsChan *__restrict__ chans, CsState *__restrict__ state,
                                                   const long long *__restrict__ n_in, int C, const float2 *in,
                                                   long long in_stride, float2 *out, unsigned long long *phase,
                                                   float *err, long long out_stride) {
    __shared__ float2 s_xz[2][32][CS_TILE + 1];
    __shared__ unsigned long long s_ph[2][32][CS_TILE + 1];
    __shared__ float s_e[2][32][CS_TILE + 1];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int ch0 = blockIdx.x * 32;
    const int my = ch0 + lane;
    const bool live = my < C;
    const long long n = live ? n_in[my] : 0;
    long long nmax = n;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
    const long long ntiles = (nmax + CS_TILE - 1) / CS_TILE;
    const int nrows = min(32, C - ch0);

    // symbols of row r in the tile at base (row r's count is lane r's n)
    auto count = [&](int r, long long base) {
        const long long nr = __shfl_sync(0xffffffffu, n, r);
        return (int)max(0ll, min((long long)CS_TILE, nr - base));
    };
    auto issue = [&](long long tile, int buf) {
        const long long base = tile * CS_TILE;
#pragma unroll 4
        for (int r = 0; r < 32; ++r)
            if (r < nrows && lane < count(r, base))
                cp_async8(&s_xz[buf][r][lane], in + (long long)(ch0 + r) * in_stride + base + lane);
        cp_async_commit();
    };

    if (role == 1 && ntiles > 0) {
        issue(0, 0);
        cp_async_wait<0>();
    }
    CsChan c{};
    CsState st{};
    if (role == 0 && live) {
        c = chans[my];
        st = state[my];
    }
    __syncthreads();
    // iteration t: warp 0 steps tile t; warp 1 stores tile t - 1 and loads tile t + 1 (both in buffer (t + 1) & 1)
    for (long long tile = 0; tile <= ntiles; ++tile) {
        const int buf = (int)(tile & 1);
        if (role == 0) {
            if (tile < ntiles) {
                const int cnt = (int)max(0ll, min((long long)CS_TILE, n - tile * CS_TILE));
                float2 *pxz = &s_xz[buf][lane][0];
                unsigned long long *pph = &s_ph[buf][lane][0];
                float *pe = &s_e[buf][lane][0];
                float2 xn = pxz[0];
                for (int i = 0; i < cnt; ++i) {
                    const float2 x = xn;
                    xn = pxz[i + 1];  // the next symbol's load leaves the dependent chain (the row has a pad element)
                    const float2 r = nco_rot_fast(st.phi);
                    const float zr = __fsub_rn(__fmul_rn(x.x, r.x), __fmul_rn(x.y, r.y));
                    const float zi = __fadd_rn(__fmul_rn(x.x, r.y), __fmul_rn(x.y, r.x));
                    const float g = cs_detector(c, zr, zi);
                    const float e = isfinite(g) ? fminf(fmaxf(g, -c.emax), c.emax) : 0.f;
                    pxz[i] = make_float2(zr, zi);
                    pph[i] = st.phi;
                    pe[i] = e;
                    st.nu = min(max(st.nu + cs_q(__fmul_rn(c.ki, e)), -c.V), c.V);
                    st.phi += (unsigned long long)(st.nu + cs_q(__fmul_rn(c.kp, e))) << 24;
                }
            }
        } else {
            const int nb = buf ^ 1;
            if (tile > 0) {
                const long long base = (tile - 1) * CS_TILE;
#pragma unroll 4
                for (int r = 0; r < 32; ++r) {
                    if (r < nrows && lane < count(r, base)) {
                        const long long at = (long long)(ch0 + r) * out_stride + base + lane;
                        out[at] = s_xz[nb][r][lane];
                        if (phase) phase[at] = s_ph[nb][r][lane];
                        if (err) err[at] = s_e[nb][r][lane];
                    }
                }
                __syncwarp();  // every lane's shared loads are done before the next tile lands in the same buffer
            }
            if (tile + 1 < ntiles) {
                issue(tile + 1, nb);
                cp_async_wait<0>();
            }
        }
        __syncthreads();
    }
    if (role == 0 && live) state[my] = st;
}

}  // namespace

struct CsyncHost {
    int dev = 0;
    size_t C = 0;
    std::vector<CsChan> chans;
    std::vector<CsState> init;         // the creation state
    bool fresh = true;                 // the device state is the creation state's once uploaded
};

struct sdr_csync : CsyncHost {
    StreamRef stream;
    DevBuf d_chans, d_state, d_n;
    std::vector<long long> n_host;
    DevBuf d_in, d_out, d_phase, d_err;

    int alloc(void *user_stream, const sdr_csync *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(CsChan), stream.s))) return rc;
        if ((rc = d_state.alloc(C * sizeof(CsState)))) return rc;
        if ((rc = d_n.alloc(C * sizeof(long long)))) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_csync &src) {
        return cuda_status(cudaMemcpy(d_state.p, src.d_state.p, C * sizeof(CsState), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_csync_t *sdr_csync_create(const sdr_csync_config_t *cfg, int *err) {
    bool ok = cfg && cfg->loops && cfg->n_channels >= 1 && cfg->n_channels <= CS_MAX_CH &&
              (cfg->n_loops == 1 || cfg->n_loops == cfg->n_channels);
    std::vector<long long> V;
    for (size_t k = 0; ok && k < cfg->n_channels; ++k) {
        const sdr_csync_loop_t &lp = cfg->loops[cfg->n_loops == 1 ? 0 : k];
        const unsigned M = lp.order;
        ok = (M == 2 || M == 4 || M == 8) && lp.kp >= 0.f && lp.ki >= 0.f && std::isfinite(lp.kp) &&
             std::isfinite(lp.ki) && lp.err_max > 0.f && std::isfinite(lp.err_max);
        if (!ok) break;
        // one correction stays below half a decision sector, 1 / (2M) turn (and q fits)
        const float sector = 1.0f / (float)(2 * M);
        ok = lp.kp * lp.err_max < sector && lp.ki * lp.err_max < sector && lp.max_freq >= 0.0 &&
             lp.max_freq <= 1.0 / (2.0 * M);
        if (!ok) break;
        V.push_back((long long)std::floor(lp.max_freq * 0x1p40));  // exact: scaling by 2^40 is exact
        ok = !cfg->freq || (cfg->freq[k] >= -V.back() && cfg->freq[k] <= V.back());
    }
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_csync>(err, cfg->device, cfg->stream, [&](sdr_csync &h) {
        const size_t C = cfg->n_channels;
        h.C = C;
        h.chans.resize(C);
        h.init.resize(C);
        for (size_t k = 0; k < C; ++k) {
            const sdr_csync_loop_t &lp = cfg->loops[cfg->n_loops == 1 ? 0 : k];
            h.chans[k] = CsChan{lp.kp, lp.ki, lp.err_max, lp.order == 8 ? 0.41421356237309503f : 1.0f, V[k],
                                lp.order == 2 ? 1 : 0, 0};
            h.init[k] = CsState{cfg->phase ? cfg->phase[k] : 0ull, cfg->freq ? (long long)cfg->freq[k] : 0ll};
        }
        return SDR_OK;
    });
}

extern "C" void sdr_csync_destroy(sdr_csync_t *h) { destroy_handle(h); }

extern "C" int sdr_csync_reset(sdr_csync_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    h->fresh = true;  // the next call uploads the creation state
    return SDR_OK;
}

extern "C" sdr_csync_t *sdr_csync_clone(const sdr_csync_t *src, int *err) { return clone_handle<CsyncHost>(src, err); }

extern "C" int sdr_csync_get_state(sdr_csync_t *h, size_t channel, uint64_t *phase, int64_t *freq) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!phase || !freq) return SDR_ERR_BAD_DATA_PTR;
    if (channel >= h->C) return SDR_ERR_INVALID_ARG;
    CsState st = h->init[channel];
    if (!h->fresh) {
        DeviceGuard g(h->dev);
        if (!g.ok) return g.status();
        SDR_CUDA_TRY(cudaMemcpyAsync(&st, (const CsState *)h->d_state.p + channel, sizeof(CsState),
                                     cudaMemcpyDeviceToHost, h->stream.s));
        SDR_CUDA_TRY(cudaStreamSynchronize(h->stream.s));
    }
    *phase = st.phi;
    *freq = st.nu;
    return SDR_OK;
}

// in: C device rows (row stride in_stride), row k of n_in[k] symbols; outputs: C rows of out_stride.  Asynchronous.
static int cs_run(sdr_csync *h, const float2 *in, const size_t *n_in, size_t in_stride, float2 *out,
                  unsigned long long *phase, float *err, size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    h->n_host.assign(n_in, n_in + C);
    if (h->fresh) {
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_state.p, h->init.data(), C * sizeof(CsState), cudaMemcpyHostToDevice, st));
        h->fresh = false;
    }
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_n.p, h->n_host.data(), C * sizeof(long long), cudaMemcpyHostToDevice, st));
    csync_kernel<<<(unsigned)((C + 31) / 32), 64, 0, st>>>((const CsChan *)h->d_chans.p, (CsState *)h->d_state.p,
                                                           (const long long *)h->d_n.p, (int)C, in,
                                                           C > 1 ? (long long)in_stride : 0, out, phase, err,
                                                           C > 1 ? (long long)out_stride : 0);
    count_launch();
    return launch_status();
}

static int cs_check(const sdr_csync *h, const float *in, const size_t *n_in, size_t in_stride, const float *out,
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

extern "C" int sdr_csync_process_dev(sdr_csync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                     float *out_c64, uint64_t *phase, float *err, size_t out_stride) {
    size_t longest = 0;
    int rc = cs_check(h, in_c64, n_in, in_stride, out_c64, out_stride, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0 || ((uintptr_t)phase % 8) != 0 ||
        ((uintptr_t)err % 4) != 0)
        return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    return cs_run(h, (const float2 *)in_c64, n_in, in_stride, (float2 *)out_c64, (unsigned long long *)phase, err,
                  out_stride);
}

extern "C" int sdr_csync_process(sdr_csync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                 float *out_c64, uint64_t *phase, float *err, size_t out_stride) {
    size_t longest = 0;
    int rc = cs_check(h, in_c64, n_in, in_stride, out_c64, out_stride, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t istride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : longest;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` symbols per channel: H2D, compute, D2H
    const size_t chunk = std::min(longest, std::max<size_t>(1, CS_HOST_BYTES / (C * 8)));
    const bool equal = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_out.reserve(chunk * C * 8);
    if (!rc && phase) rc = h->d_phase.reserve(chunk * C * 8);
    if (!rc && err) rc = h->d_err.reserve(chunk * C * 4);
    if (rc) return rc;
    std::vector<size_t> take(C);
    // one array of C rows between the host rows (stride hs, at column `at`) and the device rows (chunk apart)
    auto move = [&](void *host, size_t hs, void *dev, size_t bytes, size_t at, cudaMemcpyKind kind) -> int {
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
        if ((rc = move((void *)in_c64, istride, h->d_in.p, 8, at, cudaMemcpyHostToDevice))) return rc;
        rc = cs_run(h, (const float2 *)h->d_in.p, take.data(), chunk, (float2 *)h->d_out.p,
                    phase ? (unsigned long long *)h->d_phase.p : nullptr, err ? (float *)h->d_err.p : nullptr, chunk);
        if (rc) return rc;
        if ((rc = move(out_c64, ostride, h->d_out.p, 8, at, cudaMemcpyDeviceToHost))) return rc;
        if (phase && (rc = move(phase, ostride, h->d_phase.p, 8, at, cudaMemcpyDeviceToHost))) return rc;
        if (err && (rc = move(err, ostride, h->d_err.p, 4, at, cudaMemcpyDeviceToHost))) return rc;
    }
    return cuda_status(cudaStreamSynchronize(st));
}

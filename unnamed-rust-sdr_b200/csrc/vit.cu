// vit.cu -- K18, sdr_vit_*: Viterbi decoder bank.  C independent soft-decision streams of one rate-1/n convolutional
// code (constraint length K, S = 2^(K-1) states); sdr_b200.h states the definition in full.  Per step t of channel k:
//     q_j  = 0 for a non-finite x, else rint(clamp(fl(x[t n + j] sigma_k), -127, 127))   (half to even)
//     cost = sum_j (c_j ? 127 + q_j : 127 - q_j)
//     m'(s') = min_b m(p_b) + cost(p_b -> s'),  p_b = ((s' << 1) & (S-1)) | b;  d = 1 only when b = 1 is strictly less
// and at every step total T = 32 j >= L + 32 a traceback of L + 32 steps from the best state releases the bits of steps
// [T - L - 32, T - L).  Counts depend on T only, so the host knows them and a call copies nothing back.
// Metrics are held as u32 and compared modulo 2^32: the spread max m - min m never exceeds (2K - 3) 254 n + 1 < 2^14
// (DESIGN K18), so the sign of a 32-bit difference is the sign of the exact one and no renormalisation is needed.
// The metrics, the last L + 64 steps of decision words and T of every channel live on the device between calls.
#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"
#include "ptx.cuh"

using namespace sdr;

namespace {

constexpr size_t VIT_MAX_CH = 65536;
constexpr size_t VIT_HOST_BYTES = (size_t)32 << 20;  // host-memory calls: chunk size of input

__host__ __device__ inline long long vit_released(unsigned long long T, int L) {
    const long long t = (long long)(T & ~31ull) - L;
    return t > 0 ? t : 0;
}

// geometry of one CTA for states-per-lane SPL: G = S / SPL lanes per channel (min(S, 32)), CH = 32 / G channels,
// ring R = L + 64 steps of SPL decision words per channel (one word when S < 32), padded by one word against bank
// conflicts between channels; cost tables [2][CH][32 steps][P = 2^n] u16, padded by two entries per channel
struct VitGeom {
    int S, SPL, G, CH, R, RS, P, CS;
    __host__ __device__ VitGeom(int K, int n, int L) {
        S = 1 << (K - 1);
        SPL = S > 32 ? S / 32 : 1;
        G = S / SPL;
        CH = 32 / G;
        R = L + 64;
        RS = R * SPL + 1;
        P = 1 << n;
        CS = 32 * P + 2;
    }
    __host__ size_t smem(int n) const {
        return (size_t)CH * RS * 4 + 2 * 32 * SPL * 4 + (size_t)CH * 32 * n * 4 + 2 * CH * 4 + 2 * (size_t)CH * CS * 2;
    }
};

// A CTA of two warps owns CH channels (slots); tile t covers steps [32 (j0 + t), 32 (j0 + t) + 32) of each slot's own
// stream, j0 = floor(T0 / 32), so release points fall on tile ends whatever T0 each channel brings.
//   warp 0: a segment of G lanes per slot runs the add-compare-select, lane q owning new states j G + q (j < SPL):
//           one 8-byte load of the predecessor pair, two costs from the tile's table, a modular compare; the
//           decisions of a step are __ballot_sync words into the shared ring.  At the end of a tile it writes the
//           segment's best state (least metric, lowest index) for the traceback.
//   warp 1: traces back the PREVIOUS tile of every slot whose step total reached a release point (lane g: slot g) and
//           writes the 32 released bytes, then cp.asyncs the NEXT tile's soft values and builds its cost tables.
// One barrier per tile.  The ring holds L + 64 steps, so the traceback's L + 32 steps never meet the tile in flight.
template <int SPL>
__global__ void __launch_bounds__(64) vit_kernel(const float *__restrict__ scale, uint32_t *__restrict__ metric,
                                                 uint32_t *__restrict__ ring, unsigned long long *__restrict__ total,
                                                 const long long *__restrict__ n_in, int C, int K, int n, int L,
                                                 uint4 gens, int zero_start, int fresh, const float *in,
                                                 long long in_stride, uint8_t *out, long long out_stride) {
    extern __shared__ __align__(16) uint32_t vit_smem[];
    const VitGeom geo(K, n, L);
    const int S = geo.S, G = geo.G, CH = geo.CH, R = geo.R, RS = geo.RS, P = geo.P, CS = geo.CS;
    uint32_t *s_m = vit_smem;                               // [2][32 SPL], first: its pairs are read as 8 bytes
    uint32_t *s_ring = s_m + 2 * 32 * SPL;                  // [CH][RS]
    float *s_in = (float *)(s_ring + CH * RS);              // [CH][32 n]
    uint32_t *s_best = (uint32_t *)(s_in + CH * 32 * n);    // [2][CH]
    uint16_t *s_cost = (uint16_t *)(s_best + 2 * CH);       // [2][CH][CS]
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int ch0 = blockIdx.x * CH;
    const int nrows = min(CH, C - ch0);
    // lane r < nrows holds slot r's count and first step total
    const long long nr = lane < nrows ? n_in[ch0 + lane] : 0;
    const unsigned long long tr = lane < nrows && !fresh ? total[ch0 + lane] : 0ull;
    const int ar = (int)(tr & 31);
    long long tiles = nr > 0 ? (ar + nr + 31) / 32 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tiles = max(tiles, __shfl_xor_sync(0xffffffffu, tiles, o));
    const long long ntiles = tiles;
    const uint32_t I = zero_start ? (uint32_t)((K - 1) * 254 * n + 1) : 0u;

    // the carried ring and metrics (or the creation metrics)
    const int words = nrows * R * SPL;
    if (!fresh)
        for (int w = threadIdx.x; w < words; w += 64) {
            const int g = w / (R * SPL);
            s_ring[g * RS + (w - g * R * SPL)] = ring[(long long)ch0 * R * SPL + w];
        }
    for (int w = threadIdx.x; w < nrows * S; w += 64)
        s_m[w] = fresh ? ((w & (S - 1)) ? I : 0u) : metric[(long long)ch0 * S + w];

    const uint32_t gw[4] = {gens.x, gens.y, gens.z, gens.w};
    // warp 1: soft values of tile tt into s_in, then the cost of every code pattern at every step into buffer buf
    auto stage = [&](long long tt, int buf) {
        for (int g = 0; g < nrows; ++g) {
            const long long c = __shfl_sync(0xffffffffu, nr, g);
            const int a = __shfl_sync(0xffffffffu, ar, g);
            const long long base = (32 * tt - a) * n;  // float index of the tile's step 0 in the row
            const float *row = in + (long long)(ch0 + g) * in_stride;
            for (int e = lane; e < 32 * n; e += 32)
                if (base + e >= 0 && base + e < c * n) cp_async4(&s_in[g * 32 * n + e], row + base + e);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
        for (int g = 0; g < nrows; ++g) {
            const long long c = __shfl_sync(0xffffffffu, nr, g);
            const int a = __shfl_sync(0xffffffffu, ar, g);
            const float sc = scale[ch0 + g];
            const long long r = 32 * tt + lane - a;
            const bool act = r >= 0 && r < c;
            int q[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < n && act) {
                    const float x = s_in[g * 32 * n + lane * n + j];
                    const float v = fminf(fmaxf(__fmul_rn(x, sc), -127.f), 127.f);
                    q[j] = isfinite(x) ? __float2int_rn(v) : 0;
                }
            }
            uint16_t *cst = s_cost + (buf * CH + g) * CS + lane * P;
            for (int p = 0; p < P; ++p) {
                int v = 127 * n;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < n) v += ((p >> j) & 1) ? q[j] : -q[j];
                cst[p] = (uint16_t)v;
            }
        }
    };
    if (role == 1 && ntiles > 0) stage(0, 0);

    // warp 0: segment g = slot g, lane q of it; its code patterns per owned state and branch
    const int g = lane / G, q = lane & (G - 1);
    const long long n_g = __shfl_sync(0xffffffffu, nr, min(g, 31));
    const int a_g = __shfl_sync(0xffffffffu, ar, min(g, 31));
    uint32_t pat0[SPL], pat1[SPL];
#pragma unroll
    for (int j = 0; j < SPL; ++j) {
        const uint32_t sp = j * G + q;
        const uint32_t r0 = ((sp >> (K - 2)) << (K - 1)) | ((sp << 1) & (S - 1));
        uint32_t p0 = 0, p1 = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i < n) {
                p0 |= (uint32_t)(__popc(r0 & gw[i]) & 1) << i;
                p1 |= (uint32_t)(__popc((r0 | 1u) & gw[i]) & 1) << i;
            }
        }
        pat0[j] = p0;
        pat1[j] = p1;
    }
    __syncthreads();

    int cur = 0;  // the metric buffer of the current step (32 steps per tile: 0 at every tile boundary)
    const int R32 = R / 32;
    for (long long tile = 0; tile <= ntiles; ++tile) {
        const int buf = (int)(tile & 1);
        if (role == 0) {
            if (tile < ntiles) {
                const unsigned long long j0 = (unsigned long long)__shfl_sync(0xffffffffu, (long long)(tr >> 5), min(g, 31));
                const int sb = (int)((j0 % R32 + tile % R32) % R32) * 32;  // ring slot of the tile's step 0
                const uint16_t *cst = s_cost + (buf * CH + min(g, CH - 1)) * CS;
                uint32_t *ringg = s_ring + min(g, CH - 1) * RS;
                for (int i = 0; i < 32; ++i) {
                    const long long r = 32 * tile + i - a_g;
                    const bool act = g < nrows && r >= 0 && r < n_g;
                    const uint32_t *mo = s_m + cur * 32 * SPL + g * S;
                    uint32_t *mn = s_m + (cur ^ 1) * 32 * SPL + g * S;
                    const uint16_t *ci = cst + i * P;
                    uint32_t word[SPL];
#pragma unroll
                    for (int j = 0; j < SPL; ++j) {
                        const int sp = j * G + q;
                        const uint2 pm = *reinterpret_cast<const uint2 *>(&mo[(sp << 1) & (S - 1)]);
                        const uint32_t a0 = pm.x + ci[pat0[j]], a1 = pm.y + ci[pat1[j]];
                        const bool d = (int)(a1 - a0) < 0;
                        mn[sp] = act ? (d ? a1 : a0) : mo[sp];
                        word[j] = __ballot_sync(0xffffffffu, d);
                    }
                    if (act && q < SPL) {
                        uint32_t w = word[0];
#pragma unroll
                        for (int j = 1; j < SPL; ++j)
                            if (q == j) w = word[j];
                        if (S < 32) w = (w >> (g * S)) & ((1u << S) - 1);
                        ringg[(sb + i) * SPL + q] = w;
                    }
                    __syncwarp();
                    cur ^= 1;
                }
                // the best state after the tile's last step: least metric, ties to the lowest index
                const uint32_t *m = s_m + cur * 32 * SPL + g * S;
                uint32_t bv = m[q], bi = q;
#pragma unroll
                for (int j = 1; j < SPL; ++j) {
                    const uint32_t v = m[j * G + q];
                    if ((int)(v - bv) < 0) {
                        bv = v;
                        bi = j * G + q;
                    }
                }
                for (int o = G / 2; o > 0; o >>= 1) {
                    const uint32_t ov = __shfl_xor_sync(0xffffffffu, bv, o, G);
                    const uint32_t oi = __shfl_xor_sync(0xffffffffu, bi, o, G);
                    if ((int)(ov - bv) < 0 || (ov == bv && oi < bi)) {
                        bv = ov;
                        bi = oi;
                    }
                }
                if (q == 0 && g < nrows) s_best[buf * CH + g] = bi;
            }
        } else {
            if (tile > 0 && lane < nrows) {
                // slot `lane`: did tile - 1 end on a release point?
                const long long tt = tile - 1;
                const long long rl = 32 * tt + 31 - ar;
                const unsigned long long Tend = ((tr >> 5) + (unsigned long long)tt + 1) * 32;
                if (rl >= 0 && rl < nr && Tend >= (unsigned long long)(L + 32)) {
                    const uint32_t *rg = s_ring + lane * RS;
                    uint32_t s = s_best[(int)(tt & 1) * CH + lane];
                    int slot = (int)(((tr >> 5) % R32 + tt % R32) % R32) * 32 + 31;
                    uint32_t bits = 0;
                    for (int j = 0; j < L + 32; ++j) {
                        const uint32_t w = rg[slot * SPL + (s >> 5)];
                        if (j >= L) bits |= (s >> (K - 2)) << (L + 31 - j);
                        s = ((s << 1) & (S - 1)) | ((w >> (s & 31)) & 1u);
                        slot = slot ? slot - 1 : R - 1;
                    }
                    const long long o = (long long)Tend - L - 32 - vit_released(tr, L);
                    uint32_t *dst = reinterpret_cast<uint32_t *>(out + (long long)(ch0 + lane) * out_stride + o);
#pragma unroll
                    for (int w = 0; w < 8; ++w) {
                        const uint32_t b = bits >> (4 * w);
                        dst[w] = (b & 1u) | ((b >> 1) & 1u) << 8 | ((b >> 2) & 1u) << 16 | ((b >> 3) & 1u) << 24;
                    }
                }
            }
            if (tile + 1 < ntiles) stage(tile + 1, buf ^ 1);
        }
        __syncthreads();
    }
    for (int w = threadIdx.x; w < words; w += 64) {
        const int gg = w / (R * SPL);
        ring[(long long)ch0 * R * SPL + w] = s_ring[gg * RS + (w - gg * R * SPL)];
    }
    for (int w = threadIdx.x; w < nrows * S; w += 64) metric[(long long)ch0 * S + w] = s_m[w];
    if (threadIdx.x < nrows) total[ch0 + threadIdx.x] = tr + (unsigned long long)nr;
}

// one warp per listed channel: the remaining T - E(T) bits by a traceback from state 0 or the best state, then the
// channel's creation state
__global__ void __launch_bounds__(32) vit_finish_kernel(uint32_t *__restrict__ metric, uint32_t *__restrict__ ring,
                                                        unsigned long long *__restrict__ total,
                                                        const int *__restrict__ chans, int K, int n, int L,
                                                        int zero_start, int terminated, uint8_t *out,
                                                        long long out_stride) {
    const int S = 1 << (K - 1), SPL = S > 32 ? S / 32 : 1, R = L + 64;
    const int ch = chans[blockIdx.x], lane = threadIdx.x;
    uint32_t *m = metric + (long long)ch * S;
    const unsigned long long T = total[ch];
    uint32_t bv = m[lane & (S - 1)], bi = lane & (S - 1);
    for (int s = lane + 32; s < S; s += 32) {
        const uint32_t v = m[s];
        if ((int)(v - bv) < 0) {
            bv = v;
            bi = s;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const uint32_t ov = __shfl_xor_sync(0xffffffffu, bv, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if ((int)(ov - bv) < 0 || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    if (lane == 0) {
        const long long e = vit_released(T, L);
        const uint32_t *rg = ring + (long long)ch * R * SPL;
        uint8_t *dst = out + (long long)blockIdx.x * out_stride;
        uint32_t s = terminated ? 0u : bi;
        for (long long i = (long long)T - 1; i >= e; --i) {
            const uint32_t w = rg[(int)(i % R) * SPL + (s >> 5)];
            dst[i - e] = (uint8_t)(s >> (K - 2));
            s = ((s << 1) & (S - 1)) | ((w >> (s & 31)) & 1u);
        }
    }
    __syncwarp();
    const uint32_t I = zero_start ? (uint32_t)((K - 1) * 254 * n + 1) : 0u;
    for (int s = lane; s < S; s += 32) m[s] = s ? I : 0u;
    if (lane == 0) total[ch] = 0;
}

}  // namespace

struct VitHost {
    int dev = 0;
    int K = 0, n = 0, L = 0, zero_start = 0;
    size_t C = 0;
    uint32_t gens[4] = {0, 0, 0, 0};
    std::vector<float> scale;                // C scales
    std::vector<unsigned long long> T;       // step total per channel since create, reset or finish
    bool fresh = true;                       // the device state is the creation state's (set up by the next call)
};

struct sdr_vit : VitHost {
    StreamRef stream;
    DevBuf d_scale, d_metric, d_ring, d_total, d_n, d_chans;
    std::vector<long long> n_host;
    std::vector<int> fin_host;
    DevBuf d_in, d_out;

    size_t S() const { return (size_t)1 << (K - 1); }
    size_t ring_words() const { return C * (size_t)(L + 64) * std::max<size_t>(1, S() / 32); }
    int alloc(void *user_stream, const sdr_vit *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_scale.upload(scale.data(), C * sizeof(float), stream.s))) return rc;
        if ((rc = d_metric.alloc(C * S() * sizeof(uint32_t)))) return rc;
        if ((rc = d_ring.alloc(ring_words() * sizeof(uint32_t)))) return rc;
        if ((rc = d_total.alloc(C * sizeof(unsigned long long)))) return rc;
        if ((rc = d_n.alloc(C * sizeof(long long)))) return rc;
        if ((rc = d_chans.alloc(C * sizeof(int)))) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_vit &src) {
        SDR_CUDA_TRY(cudaMemcpy(d_metric.p, src.d_metric.p, C * S() * sizeof(uint32_t), cudaMemcpyDeviceToDevice));
        SDR_CUDA_TRY(cudaMemcpy(d_ring.p, src.d_ring.p, ring_words() * sizeof(uint32_t), cudaMemcpyDeviceToDevice));
        return cuda_status(
            cudaMemcpy(d_total.p, src.d_total.p, C * sizeof(unsigned long long), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_vit_t *sdr_vit_create(const sdr_vit_config_t *cfg, int *err) {
    bool ok = cfg && cfg->constraint >= 3 && cfg->constraint <= 9 && cfg->gens && cfg->n_gens >= 2 &&
              cfg->n_gens <= 4 && cfg->depth >= 32 && cfg->depth <= 512 && cfg->depth % 32 == 0 && cfg->scale &&
              cfg->n_channels >= 1 && cfg->n_channels <= VIT_MAX_CH &&
              (cfg->n_scales == 1 || cfg->n_scales == cfg->n_channels);
    for (size_t j = 0; ok && j < cfg->n_gens; ++j) ok = cfg->gens[j] >= 1 && cfg->gens[j] < (1u << cfg->constraint);
    for (size_t k = 0; ok && k < cfg->n_scales; ++k) ok = cfg->scale[k] > 0.f && std::isfinite(cfg->scale[k]);
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_vit>(err, cfg->device, cfg->stream, [&](sdr_vit &h) {
        h.K = (int)cfg->constraint;
        h.n = (int)cfg->n_gens;
        h.L = (int)cfg->depth;
        h.zero_start = cfg->zero_start ? 1 : 0;
        h.C = cfg->n_channels;
        for (size_t j = 0; j < cfg->n_gens; ++j) h.gens[j] = cfg->gens[j];
        h.scale.resize(h.C);
        for (size_t k = 0; k < h.C; ++k) h.scale[k] = cfg->scale[cfg->n_scales == 1 ? 0 : k];
        h.T.assign(h.C, 0);
        return SDR_OK;
    });
}

extern "C" void sdr_vit_destroy(sdr_vit_t *h) { destroy_handle(h); }

extern "C" int sdr_vit_reset(sdr_vit_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    h->fresh = true;  // the next call starts every channel from the creation metrics at T = 0
    std::fill(h->T.begin(), h->T.end(), 0ull);
    return SDR_OK;
}

extern "C" sdr_vit_t *sdr_vit_clone(const sdr_vit_t *src, int *err) { return clone_handle<VitHost>(src, err); }

extern "C" int sdr_vit_output_count(const sdr_vit_t *h, const size_t *n_in, size_t *n_out) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !n_out) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k)
        n_out[k] = (size_t)(vit_released(h->T[k] + n_in[k], h->L) - vit_released(h->T[k], h->L));
    return SDR_OK;
}

// in: C device rows of n_in[k] steps (n floats each, row stride in_stride steps); out: C rows of out_stride bytes.
// Asynchronous.
static int vit_run(sdr_vit *h, const float *in, const size_t *n_in, size_t in_stride, uint8_t *out,
                   size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    h->n_host.assign(n_in, n_in + C);
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_n.p, h->n_host.data(), C * sizeof(long long), cudaMemcpyHostToDevice, st));
    const VitGeom geo(h->K, h->n, h->L);
    const unsigned grid = (unsigned)((C + geo.CH - 1) / geo.CH);
    const size_t smem = geo.smem(h->n);
    const uint4 g = make_uint4(h->gens[0], h->gens[1], h->gens[2], h->gens[3]);
    const long long is = C > 1 ? (long long)in_stride * h->n : 0, os = C > 1 ? (long long)out_stride : 0;
#define VIT_ARGS                                                                                                   \
    (const float *)h->d_scale.p, (uint32_t *)h->d_metric.p, (uint32_t *)h->d_ring.p,                               \
        (unsigned long long *)h->d_total.p, (const long long *)h->d_n.p, (int)C, h->K, h->n, h->L, g, h->zero_start, \
        h->fresh ? 1 : 0, in, is, out, os
    switch (geo.SPL) {
    case 1: vit_kernel<1><<<grid, 64, smem, st>>>(VIT_ARGS); break;
    case 2: vit_kernel<2><<<grid, 64, smem, st>>>(VIT_ARGS); break;
    case 4: vit_kernel<4><<<grid, 64, smem, st>>>(VIT_ARGS); break;
    default: vit_kernel<8><<<grid, 64, smem, st>>>(VIT_ARGS); break;
    }
#undef VIT_ARGS
    count_launch();
    h->fresh = false;
    for (size_t k = 0; k < C; ++k) h->T[k] += n_in[k];
    return launch_status();
}

// the counts of a call, and the checks every process call makes; *longest: the longest input row
static int vit_check(sdr_vit *h, const float *in, const size_t *n_in, size_t in_stride, const uint8_t *out,
                     size_t out_stride, size_t *n_out, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !n_out) return SDR_ERR_BAD_DATA_PTR;
    *longest = *std::max_element(n_in, n_in + h->C);
    sdr_vit_output_count(h, n_in, n_out);
    if (*longest == 0) return SDR_OK;
    const size_t most = *std::max_element(n_out, n_out + h->C);
    if (!in || (most && !out)) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && (in_stride < *longest || out_stride < most)) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_vit_process_dev(sdr_vit_t *h, const float *in, const size_t *n_in, size_t in_stride, uint8_t *out,
                                   size_t out_stride, size_t *n_out) {
    size_t longest = 0;
    int rc = vit_check(h, in, n_in, in_stride, out, out_stride, n_out, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in % 4) != 0 || ((uintptr_t)out % 4) != 0 || (h->C > 1 && out_stride % 4 != 0))
        return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    return vit_run(h, in, n_in, in_stride, out, out_stride);
}

extern "C" int sdr_vit_process(sdr_vit_t *h, const float *in, const size_t *n_in, size_t in_stride, uint8_t *out,
                               size_t out_stride, size_t *n_out) {
    size_t longest = 0;
    int rc = vit_check(h, in, n_in, in_stride, out, out_stride, n_out, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C, n = (size_t)h->n;
    const size_t istride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : 0;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` steps per channel (a multiple of 32): H2D, decode, D2H
    const size_t chunk = std::min((longest + 31) & ~(size_t)31,
                                  std::max<size_t>(32, VIT_HOST_BYTES / (C * n * 4) & ~(size_t)31));
    const size_t ocap = chunk + 32;  // the most bits a round of `chunk` steps releases, rounded to a multiple of 4
    if ((rc = h->d_in.reserve(chunk * C * n * 4))) return rc;
    if ((rc = h->d_out.reserve(ocap * C))) return rc;
    std::vector<size_t> take(C), got(C), done(C, 0);
    for (size_t at = 0; at < longest; at += chunk) {
        for (size_t k = 0; k < C; ++k) {
            take[k] = n_in[k] > at ? std::min(chunk, n_in[k] - at) : 0;
            if (take[k])
                SDR_CUDA_TRY(cudaMemcpyAsync((char *)h->d_in.p + k * chunk * n * 4, in + (k * istride + at) * n,
                                             take[k] * n * 4, cudaMemcpyHostToDevice, st));
        }
        sdr_vit_output_count(h, take.data(), got.data());
        if ((rc = vit_run(h, (const float *)h->d_in.p, take.data(), chunk, (uint8_t *)h->d_out.p, ocap))) return rc;
        for (size_t k = 0; k < C; ++k) {
            if (got[k])
                SDR_CUDA_TRY(cudaMemcpyAsync(out + k * ostride + done[k], (char *)h->d_out.p + k * ocap, got[k],
                                             cudaMemcpyDeviceToHost, st));
            done[k] += got[k];
        }
    }
    return cuda_status(cudaStreamSynchronize(st));
}

// the channels a finish applies to and their counts; *most: the largest count
static int vit_finish_check(sdr_vit *h, const uint8_t *which, const uint8_t *out, size_t out_stride, size_t *n_out,
                            size_t *most) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    *most = 0;
    for (size_t k = 0; k < h->C; ++k) {
        n_out[k] = (!which || which[k]) ? (size_t)(h->T[k] - vit_released(h->T[k], h->L)) : 0;
        *most = std::max(*most, n_out[k]);
    }
    if (*most && !out) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && out_stride < *most) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

// listed channel i (in channel order) gets row i of out at row_stride bytes; asynchronous
static int vit_finish_run(sdr_vit *h, const uint8_t *which, int terminated, uint8_t *out, size_t row_stride) {
    cudaStream_t st = h->stream.s;
    h->fin_host.clear();
    for (size_t k = 0; k < h->C; ++k)
        if (!which || which[k]) h->fin_host.push_back((int)k);
    const size_t nf = h->fin_host.size();
    if (nf == 0 || h->fresh) return SDR_OK;
    SDR_CUDA_TRY(cudaMemcpyAsync(h->d_chans.p, h->fin_host.data(), nf * sizeof(int), cudaMemcpyHostToDevice, st));
    vit_finish_kernel<<<(unsigned)nf, 32, 0, st>>>((uint32_t *)h->d_metric.p, (uint32_t *)h->d_ring.p,
                                                   (unsigned long long *)h->d_total.p, (const int *)h->d_chans.p, h->K,
                                                   h->n, h->L, h->zero_start, terminated, out,
                                                   (long long)row_stride);
    count_launch();
    return launch_status();
}

extern "C" int sdr_vit_finish_dev(sdr_vit_t *h, const uint8_t *which, int terminated, uint8_t *out,
                                  size_t out_stride, size_t *n_out) {
    size_t most = 0;
    int rc = vit_finish_check(h, which, out, out_stride, n_out, &most);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    // the finish kernel writes listed channel i at row i: move the rows to the caller's channel rows through scratch
    // unless every channel is listed
    const bool all = !which || std::all_of(which, which + h->C, [](uint8_t v) { return v != 0; });
    const size_t stride = h->C > 1 ? out_stride : 0;
    if (all) {
        rc = vit_finish_run(h, nullptr, terminated, out, stride);
    } else {
        const size_t cap = (size_t)h->L + 32;
        if ((rc = h->d_out.reserve(cap * h->C))) return rc;
        if ((rc = vit_finish_run(h, which, terminated, (uint8_t *)h->d_out.p, cap))) return rc;
        size_t i = 0;
        for (size_t k = 0; k < h->C; ++k) {
            if (!which[k]) continue;
            if (n_out[k])
                SDR_CUDA_TRY(cudaMemcpyAsync(out + k * stride, (uint8_t *)h->d_out.p + i * cap, n_out[k],
                                             cudaMemcpyDeviceToDevice, h->stream.s));
            ++i;
        }
    }
    if (rc) return rc;
    for (size_t k = 0; k < h->C; ++k)
        if (!which || which[k]) h->T[k] = 0;
    return SDR_OK;
}

extern "C" int sdr_vit_finish(sdr_vit_t *h, const uint8_t *which, int terminated, uint8_t *out, size_t out_stride,
                              size_t *n_out) {
    size_t most = 0;
    int rc = vit_finish_check(h, which, out, out_stride, n_out, &most);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t cap = (size_t)h->L + 32, stride = h->C > 1 ? out_stride : 0;
    if ((rc = h->d_out.reserve(cap * h->C))) return rc;
    if ((rc = vit_finish_run(h, which, terminated, (uint8_t *)h->d_out.p, cap))) return rc;
    size_t i = 0;
    for (size_t k = 0; k < h->C; ++k) {
        if (which && !which[k]) continue;
        if (n_out[k])
            SDR_CUDA_TRY(cudaMemcpyAsync(out + k * stride, (uint8_t *)h->d_out.p + i * cap, n_out[k],
                                         cudaMemcpyDeviceToHost, h->stream.s));
        ++i;
    }
    for (size_t k = 0; k < h->C; ++k)
        if (!which || which[k]) h->T[k] = 0;
    return cuda_status(cudaStreamSynchronize(h->stream.s));
}

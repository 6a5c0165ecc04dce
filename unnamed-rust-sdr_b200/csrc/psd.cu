// psd.cu -- K8, sdr_psd_*: averaged power spectra of one IQ stream, the chain
//     window -> decimate -> map(fft::fft) -> |.|^2 -> mean of K
// Frame j holds the N samples ending at input sample (j+1) H - 1 (Window + Decimate, adapters/mod.rs:271-303,
// 14-41; x[<0] = 0), tapered by w; output g is P_g[k] = (1/K) sum_{j = gK}^{gK+K-1} |X_j[k]|^2.
// Summation order (what makes every blocking give the same bits): group g is cut into chunks of PSD_S consecutive
// frames anchored on its first frame; a chunk sums |X_j[k]|^2 in f32 in ascending j (two FMAs per bin and frame),
// the chunk partials of a group are summed in f64 in chunk order, scaled once in f64 and rounded to f32.
//   path 2 (N = 1024, u8 / c64): psd1024_kernel -- the 1024-point warp FFT of fft1024_warp_kernel with the taper on the
//           unpack and |X|^2 accumulated in 32 registers per lane instead of storing X; one partial row per chunk
//           (the final row when a group is one chunk), then psd_reduce_kernel.
//   path 1 (anything else): gather + taper frames into L2-sized slabs, the sdr_fft plan, psd_accum_kernel,
//           psd_reduce_kernel.
// Carried across calls: the samples of the frames not yet in a finished chunk, the open group's f64 accumulator and the
// stream position.  The carried tail and the new block are read through two pointers, so the block is never copied.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"
#include "fft_core.cuh"
#include "ptx.cuh"

using namespace sdr;

namespace sdr {
namespace {

constexpr long long PSD_S = 32;                      // frames per chunk (part of the definition)
constexpr size_t PSD_SLAB_BYTES = (size_t)32 << 20;  // path 1: c64 frames per slab, so the FFT's traffic stays in L2
constexpr long long PSD_PART_CHUNKS = 8192;          // path 2: chunk partials per launch (32 MiB)
constexpr unsigned PSD_FLAGS = SDR_PSD_SHIFT | SDR_PSD_NORM | SDR_PSD_GENERAL_KERNEL;

// Stream sample i of one call: 0 for i < 0 (the deque's initial zeros), hist[i - hist_lo] below in_lo (the carried
// tail), in[i - in_lo] from in_lo on.  Only frames complete in [.., end) are read.
struct PsdSrc {
    const void *hist;
    const void *in;
    long long hist_lo, in_lo, end;
};

template <bool U8>
__device__ __forceinline__ float2 psd_load(const PsdSrc &s, long long i) {
    if (i < 0) return make_float2(0.f, 0.f);
    const bool h = i < s.in_lo;
    const void *base = h ? s.hist : s.in;
    const long long k = h ? i - s.hist_lo : i - s.in_lo;
    if (U8) return unpack_iq_u16(__ldg(reinterpret_cast<const uint16_t *>(base) + k));
    return __ldg(reinterpret_cast<const float2 *>(base) + k);
}

// chunk `gid` (chunks numbered across groups, cpg = ceil(K / S) per group): its first frame and frame count
__host__ __device__ __forceinline__ void psd_chunk(long long gid, long long K, long long cpg, long long *f0, long long *nf) {
    const long long g = gid / cpg, c = gid - g * cpg;
    *f0 = g * K + c * PSD_S;
    *nf = (K - c * PSD_S) < PSD_S ? K - c * PSD_S : PSD_S;
}

// |x|^2 added to a chunk sum: the same two roundings on both paths
__device__ __forceinline__ float psd_add(float acc, float2 x) { return __fmaf_rn(x.y, x.y, __fmaf_rn(x.x, x.x, acc)); }

// ---- path 2: N = 1024 ----------------------------------------------------------------------------------------------
constexpr int P1K_WARPS = 8;          // 2 CTAs (16 warps) per SM, as fft1024_warp_kernel
constexpr int P1K_XCH = 33 * 32;      // padded exchange, float2 per warp
__host__ __device__ constexpr size_t p1k_raw_offset() { return (size_t)(31 * 32 + P1K_WARPS * P1K_XCH) * sizeof(float2) + 1024 * sizeof(float); }
__host__ __device__ constexpr size_t p1k_smem(int fmt) { return p1k_raw_offset() + (fmt == SDR_FMT_U8IQ ? P1K_WARPS * 4096 : 0); }

struct Psd1kArgs {
    PsdSrc src;
    const float2 *tw;     // W_1024^k
    const float *taper;   // 1024
    long long H, K, cpg;
    long long gid0, nchunks;
    float *part;          // nchunks rows of 1024 (cpg > 1)
    float *out;           // nchunks rows of out_stride (cpg == 1: every chunk is a whole group)
    long long out_stride;
    double scale;
};

// One persistent warp per chunk at a time, frames in ascending order.  Per frame: 1024 samples from (j+1) H - N -- for
// u8 one cp.async.bulk of 2 KB into a per-warp double buffer (prefetched one frame ahead, completing on an mbarrier) when
// the frame lies in the new block at a 16-byte aligned address, per-lane loads otherwise (frames touching x[<0] or the
// carried tail, odd hops); c64 always per-lane loads, as fft1024_warp_kernel.  Both loaders give the same floats, so
// the bits do not depend on the block's address.  Taper, two radix-32 passes, then |X|^2 into acc[s] = bin lane + 32 s.
template <int FMT, bool SHIFT>
__global__ void __launch_bounds__(P1K_WARPS * 32, 2) psd1024_kernel(Psd1kArgs a) {
    constexpr int N = 1024;
    constexpr bool U8 = FMT == SDR_FMT_U8IQ;
    extern __shared__ float4 smem4[];
    __shared__ __align__(8) uint64_t tma_bar[P1K_WARPS][2];
    float2 *tw_s = reinterpret_cast<float2 *>(smem4);
    float2 *xch_all = tw_s + 31 * 32;
    float *tap_s = reinterpret_cast<float *>(xch_all + P1K_WARPS * P1K_XCH);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float2 *xch = xch_all + warp * P1K_XCH;
    unsigned char *raw = reinterpret_cast<unsigned char *>(smem4) + p1k_raw_offset() + warp * 4096;
    for (int idx = tid; idx < 31 * 32; idx += P1K_WARPS * 32) tw_s[idx] = __ldg(a.tw + (idx / 32 + 1) * (idx % 32));
    for (int idx = tid; idx < N; idx += P1K_WARPS * 32) tap_s[idx] = __ldg(a.taper + idx);
    __syncthreads();
    const long long nwarps = (long long)gridDim.x * P1K_WARPS;
    long long c = (long long)blockIdx.x * P1K_WARPS + warp;
    if (c >= a.nchunks) return;
    const unsigned char *in8 = reinterpret_cast<const unsigned char *>(a.src.in);
    // u8 frames starting at stream index s take the bulk copy when s - in_lo >= 0 and 2 (s - in_lo) + in8 = 0 mod 16
    const uint32_t in_mis = (uint32_t)reinterpret_cast<uintptr_t>(in8) & 15u;
    auto bulk = [&](long long s) { return U8 && s >= a.src.in_lo && ((in_mis + 2u * (uint32_t)(s - a.src.in_lo)) & 15u) == 0; };
    int buf = 0;
    uint32_t tph = 0;  // bit i = parity of buffer i's mbarrier
    const uint32_t bar_s = smem_u32(&tma_bar[warp][0]);
    const uint32_t raw_s = smem_u32(raw);
    auto tma_load = [&](long long s, int bf) {  // lane 0 only
        mbar_arrive_expect_tx(bar_s + 8u * bf, 2048);
        tma_bulk_g2s(raw_s + 2048u * bf, in8 + 2 * (s - a.src.in_lo), 2048, bar_s + 8u * bf);
    };
    // the current frame: number i of nf in chunk c, first sample s0
    long long f0, nfl, s0;
    psd_chunk(a.gid0 + c, a.K, a.cpg, &f0, &nfl);
    s0 = (f0 + 1) * a.H - N;
    int i = 0, nf = (int)nfl;
    if (U8) {
        if (lane == 0) {
            mbar_init(bar_s, 1);
            mbar_init(bar_s + 8u, 1);
            mbar_init_fence();
            if (bulk(s0)) tma_load(s0, 0);
        }
        __syncwarp();
    }
    float acc[32];
#pragma unroll
    for (int s = 0; s < 32; ++s) acc[s] = 0.f;
    while (true) {
        float2 v[32], w[32];
        if (U8) {
            // the next frame of the warp's sequence; buffer buf ^ 1 was last read one frame ago, before that frame's
            // closing __syncwarp
            if (lane == 0) {
                long long ns = s0 + a.H;
                bool more = true;
                if (i + 1 == nf) {
                    more = c + nwarps < a.nchunks;
                    if (more) {
                        long long g0, gn;
                        psd_chunk(a.gid0 + c + nwarps, a.K, a.cpg, &g0, &gn);
                        ns = (g0 + 1) * a.H - N;
                    }
                }
                if (more && bulk(ns)) tma_load(ns, buf ^ 1);
            }
            if (bulk(s0)) {
                mbar_wait(bar_s + 8u * buf, (tph >> buf) & 1u);
                tph ^= 1u << buf;
                const unsigned short *r16 = reinterpret_cast<const unsigned short *>(raw + buf * 2048);
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const unsigned h = r16[lane + 32 * e];
                    const unsigned mi = __byte_perm(h, 0x4B000000u, 0x7540u), mq = __byte_perm(h, 0x4B000000u, 0x7541u);
                    v[e] = make_float2(__fmaf_rn(__uint_as_float(mi), 0.0078125f, -65537.0f),
                                       __fmaf_rn(__uint_as_float(mq), 0.0078125f, -65537.0f));
                }
            } else {
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = psd_load<true>(a.src, s0 + lane + 32 * e);
            }
            buf ^= 1;
        } else {
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = psd_load<false>(a.src, s0 + lane + 32 * e);
        }
#pragma unroll
        for (int e = 0; e < 32; ++e) {
            const float t = tap_s[lane + 32 * e];
            v[e].x *= t;
            v[e].y *= t;
        }
        dft32<U8>(v, w);
#pragma unroll
        for (int s = 0; s < 32; ++s) xch[33 * lane + s] = w[s];
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = xch[lane + 33 * e];
#pragma unroll
        for (int q = 1; q < 32; ++q) v[q] = cmul(v[q], tw_s[(q - 1) * 32 + lane]);
        dft32<U8>(v, w);
#pragma unroll
        for (int s = 0; s < 32; ++s) acc[s] = psd_add(acc[s], w[s]);
        __syncwarp();
        if (++i < nf) {
            s0 += a.H;
            continue;
        }
        // chunk done.  Bin lane + 32 s lands in slot lane + 32 (s ^ 16) when shifted.
        if (a.cpg == 1) {
            float *dst = a.out + c * a.out_stride + lane;
#pragma unroll
            for (int s = 0; s < 32; ++s) dst[32 * (SHIFT ? (s ^ 16) : s)] = (float)((double)acc[s] * a.scale);
        } else {
            float *dst = a.part + c * N + lane;
#pragma unroll
            for (int s = 0; s < 32; ++s) dst[32 * (SHIFT ? (s ^ 16) : s)] = acc[s];
        }
#pragma unroll
        for (int s = 0; s < 32; ++s) acc[s] = 0.f;
        c += nwarps;
        if (c >= a.nchunks) break;
        psd_chunk(a.gid0 + c, a.K, a.cpg, &f0, &nfl);
        s0 = (f0 + 1) * a.H - N;
        i = 0;
        nf = (int)nfl;
    }
}

// ---- path 1 --------------------------------------------------------------------------------------------------------
// frames f0 .. f0 + nf - 1, tapered, side by side as c64 (the FFT plan's input)
template <bool U8>
__global__ void psd_gather_kernel(PsdSrc src, const float *__restrict__ taper, long long N, long long H, long long f0,
                                  long long nf, float2 *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float t = __ldg(taper + i);
    for (long long f = blockIdx.y; f < nf; f += gridDim.y) {
        const float2 v = psd_load<U8>(src, (f0 + f + 1) * H - N + i);
        out[f * N + i] = make_float2(v.x * t, v.y * t);
    }
}

// partial of chunk gidA + c = sum over its frames, ascending, of |y|^2 (y: spectra of frames fA ..)
__global__ void psd_accum_kernel(const float2 *__restrict__ y, long long N, long long fA, long long gidA, long long nch,
                                 long long K, long long cpg, float *__restrict__ part) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    for (long long c = blockIdx.y; c < nch; c += gridDim.y) {
        long long f0, nf;
        psd_chunk(gidA + c, K, cpg, &f0, &nf);
        float p = 0.f;
        for (long long j = f0; j < f0 + nf; ++j) p = psd_add(p, y[(j - fA) * N + k]);
        part[c * N + k] = p;
    }
}

// ---- both paths: chunk partials of chunks gidA .. gidB - 1 -> groups ------------------------------------------------
// A group whose first chunks came before gidA continues from acc_in; a group still open at gidB leaves its sum in
// acc_out (a different buffer: the group reading acc_in and the one writing acc_out may run concurrently).
__global__ void psd_reduce_kernel(const float *__restrict__ part, long long gidA, long long gidB, long long cpg,
                                  long long row_base, long long N, double scale, const double *__restrict__ acc_in,
                                  double *__restrict__ acc_out, float *__restrict__ out, long long out_stride) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    const long long gA = gidA / cpg, gB = (gidB - 1) / cpg;
    for (long long g = gA + blockIdx.y; g <= gB; g += gridDim.y) {
        const long long lo = max(gidA, g * cpg), hi = min(gidB, (g + 1) * cpg);
        double s = lo != g * cpg ? acc_in[k] : 0.0;
        for (long long c = lo; c < hi; ++c) s += (double)part[(c - gidA) * N + k];
        if (hi == (g + 1) * cpg) out[(g - row_base) * out_stride + k] = (float)(s * scale);
        else acc_out[k] = s;
    }
}

}  // namespace
}  // namespace sdr

struct PsdHost {
    int dev = 0;
    long long N = 0, H = 0, K = 0, cpg = 1;
    int fmt = SDR_FMT_C64;
    unsigned flags = 0;
    bool fused = false;          // path 2
    double scale = 1.0;          // 1/K, and 1/N with NORM
    std::vector<float> taper;
    long long total = 0;         // input samples seen
    long long done = 0;          // frames in finished chunks (a chunk boundary)
    long long hist_lo = 0;       // d_hist[cur] holds stream samples hist_lo .. total - 1
    int last_path = 0;
};

static size_t psd_es(const PsdHost *h) { return h->fmt == SDR_FMT_U8IQ ? 2 : 8; }

struct sdr_psd : PsdHost {
    StreamRef stream;
    Owned<sdr_fft_t, sdr_fft_destroy> plan;  // path 1
    DevBuf d_taper;
    DevBuf d_tw;                 // W_1024 (path 2)
    DevBuf d_hist[2];
    int cur = 0;
    DevBuf d_acc[2];             // f64 sum of the open group's finished chunks
    int acur = 0;
    DevBuf d_part, d_x, d_y, d_in, d_out;

    // taper, twiddles or FFT plan, history and accumulators of a handle whose geometry fields are set
    int alloc(void *user_stream, const sdr_psd *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        cudaStream_t st = stream.s;
        if ((rc = d_taper.upload(taper.data(), taper.size() * sizeof(float), st))) return rc;
        std::vector<float2> tw;
        if (fused) {
            // the FFT plans' table: f64 angles rounded to f32
            tw.resize(1024);
            for (int k = 0; k < 1024; ++k)
                tw[k] = make_float2((float)std::cos(-2.0 * M_PI / 1024.0 * k), (float)std::sin(-2.0 * M_PI / 1024.0 * k));
            if ((rc = d_tw.upload(tw.data(), tw.size() * sizeof(float2), st))) return rc;
        } else {
            sdr_fft_config_t fc;
            fc.n = (size_t)N;
            fc.input_format = SDR_FMT_C64;  // the gather unpacks and tapers
            fc.flags = (flags & SDR_PSD_SHIFT) ? SDR_FFT_SHIFT : 0u;  // NORM is applied in f64 at the end
            fc.device = dev;
            fc.stream = (void *)st;
            plan.reset(sdr_fft_create(&fc, &rc));
            if (!plan) return rc;
        }
        for (int i = 0; i < 2; ++i) {
            rc = d_hist[i].reserve(16);
            if (!rc) rc = d_acc[i].reserve((size_t)N * sizeof(double));
            if (rc) return rc;
        }
        return cuda_status(cudaStreamSynchronize(st));
    }
    // the history tail and the open group's accumulator
    int copy_device(const sdr_psd &src) {
        const size_t tail = (size_t)(total - hist_lo) * psd_es(this);
        int rc = SDR_OK;
        if (tail > 0) {
            rc = d_hist[0].reserve(tail);
            if (!rc) rc = cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, tail, cudaMemcpyDeviceToDevice));
        }
        if (!rc)
            rc = cuda_status(cudaMemcpy(d_acc[0].p, src.d_acc[src.acur].p, (size_t)N * sizeof(double),
                                        cudaMemcpyDeviceToDevice));
        return rc;
    }
};

extern "C" sdr_psd_t *sdr_psd_create(const sdr_psd_config_t *cfg, int *err) {
    if (!cfg || cfg->n == 0 || cfg->n > ((size_t)1 << 26) || cfg->hop == 0 || cfg->hop > ((size_t)1 << 40) ||
        cfg->average == 0 || cfg->average > ((size_t)1 << 40) ||
        (cfg->input_format != SDR_FMT_U8IQ && cfg->input_format != SDR_FMT_C64) || (cfg->flags & ~PSD_FLAGS))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_psd>(err, cfg->device, cfg->stream, [&](sdr_psd &h) {
        h.N = (long long)cfg->n;
        h.H = (long long)cfg->hop;
        h.K = (long long)cfg->average;
        h.cpg = (h.K + PSD_S - 1) / PSD_S;
        h.fmt = cfg->input_format;
        h.flags = cfg->flags;
        h.fused = h.N == 1024 && !(h.flags & SDR_PSD_GENERAL_KERNEL);
        h.scale = 1.0 / (double)h.K;
        if (h.flags & SDR_PSD_NORM) h.scale /= (double)h.N;
        h.taper.assign((size_t)h.N, 1.0f);
        if (cfg->window) std::memcpy(h.taper.data(), cfg->window, (size_t)h.N * sizeof(float));
        return SDR_OK;
    });
}

extern "C" void sdr_psd_destroy(sdr_psd_t *h) { destroy_handle(h); }

extern "C" int sdr_psd_reset(sdr_psd_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // indices below 0 read as zero and a group starting at a chunk boundary 0 never reads the accumulator
    h->total = h->done = h->hist_lo = 0;
    h->cur = h->acur = 0;
    h->last_path = 0;
    return SDR_OK;
}

extern "C" sdr_psd_t *sdr_psd_clone(const sdr_psd_t *src, int *err) { return clone_handle<PsdHost>(src, err); }

// spectra that the next n_in samples complete: frame j needs input sample (j + 1) H - 1, group g frames gK .. gK + K - 1
extern "C" size_t sdr_psd_output_count(const sdr_psd_t *h, size_t n_in) {
    if (!h) return 0;
    return (size_t)(((h->total + (long long)n_in) / h->H) / h->K - (h->total / h->H) / h->K);
}

extern "C" int sdr_psd_last_path(const sdr_psd_t *h) { return h ? h->last_path : 0; }

// chunk number of chunk boundary P (a frame index)
static long long psd_gid(const sdr_psd *h, long long P) { return (P / h->K) * h->cpg + (P % h->K) / PSD_S; }
static long long psd_frame(const sdr_psd *h, long long gid) {
    long long f0, nf;
    psd_chunk(gid, h->K, h->cpg, &f0, &nf);
    return f0;
}

static int psd_reduce(sdr_psd *h, const float *part, long long gidA, long long gidB, long long row_base, float *out,
                      size_t out_stride) {
    const long long groups = (gidB - 1) / h->cpg - gidA / h->cpg + 1;
    dim3 grid((unsigned)((h->N + 255) / 256), (unsigned)std::min<long long>(groups, 65535));
    psd_reduce_kernel<<<grid, 256, 0, h->stream.s>>>(part, gidA, gidB, h->cpg, row_base, h->N, h->scale,
                                                      (const double *)h->d_acc[h->acur].p, (double *)h->d_acc[h->acur ^ 1].p,
                                                      out, (long long)out_stride);
    count_launch();
    int rc = launch_status();
    if (rc) return rc;
    if (gidB % h->cpg != 0) h->acur ^= 1;  // the group open at gidB left its sum in the other buffer
    return SDR_OK;
}

template <int FMT, bool SHIFT>
static int psd_launch_1k(const Psd1kArgs &a, cudaStream_t st) {
    auto kern = psd1024_kernel<FMT, SHIFT>;
    const size_t smem = p1k_smem(FMT);
    SDR_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long ctas = std::min<long long>((a.nchunks + P1K_WARPS - 1) / P1K_WARPS, 2LL * current_sm_count());
    kern<<<(unsigned)ctas, P1K_WARPS * 32, smem, st>>>(a);
    count_launch();
    return launch_status();
}

static int psd_run_fused(sdr_psd *h, const PsdSrc &src, long long gid0, long long gid1, long long row_base, float *out,
                         size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const bool shift = (h->flags & SDR_PSD_SHIFT) != 0;
    const long long step = h->cpg == 1 ? gid1 - gid0 : PSD_PART_CHUNKS;
    if (h->cpg > 1) {
        const int rc = h->d_part.reserve((size_t)std::min(step, gid1 - gid0) * 1024 * sizeof(float));
        if (rc) return rc;
    }
    for (long long gA = gid0; gA < gid1; gA += step) {
        const long long gB = std::min(gid1, gA + step);
        Psd1kArgs a;
        a.src = src; a.tw = (const float2 *)h->d_tw.p; a.taper = (const float *)h->d_taper.p;
        a.H = h->H; a.K = h->K; a.cpg = h->cpg;
        a.gid0 = gA; a.nchunks = gB - gA; a.part = (float *)h->d_part.p;
        a.out = out + (gA - row_base) * (long long)out_stride;  // cpg == 1: chunk gid is group gid
        a.out_stride = (long long)out_stride; a.scale = h->scale;
        int rc = h->fmt == SDR_FMT_U8IQ ? (shift ? psd_launch_1k<SDR_FMT_U8IQ, true>(a, st) : psd_launch_1k<SDR_FMT_U8IQ, false>(a, st))
                                        : (shift ? psd_launch_1k<SDR_FMT_C64, true>(a, st) : psd_launch_1k<SDR_FMT_C64, false>(a, st));
        if (rc) return rc;
        if (h->cpg > 1) {
            rc = psd_reduce(h, (const float *)h->d_part.p, gA, gB, row_base, out, out_stride);
            if (rc) return rc;
        }
    }
    return SDR_OK;
}

static int psd_run_general(sdr_psd *h, const PsdSrc &src, long long gid0, long long gid1, long long row_base,
                           float *out, size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const long long N = h->N;
    // whole chunks per slab: about PSD_SLAB_BYTES of frames, at least one chunk
    const long long cap = std::max<long long>(1, (long long)(PSD_SLAB_BYTES / ((size_t)N * 8)));
    const long long step = std::max<long long>(1, cap / std::min(h->K, PSD_S));
    const long long max_frames = std::min(step, gid1 - gid0) * std::min(h->K, PSD_S);
    int rc = h->d_x.reserve((size_t)max_frames * N * 8);
    if (!rc) rc = h->d_y.reserve((size_t)max_frames * N * 8);
    if (!rc) rc = h->d_part.reserve((size_t)std::min(step, gid1 - gid0) * N * sizeof(float));
    if (rc) return rc;
    for (long long gA = gid0; gA < gid1; gA += step) {
        const long long gB = std::min(gid1, gA + step);
        const long long fA = psd_frame(h, gA), nf = psd_frame(h, gB) - fA;
        dim3 grid((unsigned)((N + 255) / 256), (unsigned)std::min<long long>(nf, 65535));
        if (h->fmt == SDR_FMT_U8IQ)
            psd_gather_kernel<true><<<grid, 256, 0, st>>>(src, (const float *)h->d_taper.p, N, h->H, fA, nf, (float2 *)h->d_x.p);
        else
            psd_gather_kernel<false><<<grid, 256, 0, st>>>(src, (const float *)h->d_taper.p, N, h->H, fA, nf, (float2 *)h->d_x.p);
        count_launch();
        rc = launch_status();
        if (!rc) rc = sdr_fft_exec_dev(h->plan.get(), h->d_x.p, (size_t)nf, (float *)h->d_y.p);
        if (rc) return rc;
        grid.y = (unsigned)std::min<long long>(gB - gA, 65535);
        psd_accum_kernel<<<grid, 256, 0, st>>>((const float2 *)h->d_y.p, N, fA, gA, gB - gA, h->K, h->cpg, (float *)h->d_part.p);
        count_launch();
        rc = launch_status();
        if (!rc) rc = psd_reduce(h, (const float *)h->d_part.p, gA, gB, row_base, out, out_stride);
        if (rc) return rc;
    }
    return SDR_OK;
}

// in: n_in device samples; out: the spectra the call completes, rows of out_stride floats
static int psd_run(sdr_psd *h, const void *in, size_t n_in, float *out, size_t out_stride) {
    cudaStream_t st = h->stream.s;
    const size_t es = psd_es(h);
    const long long end = h->total + (long long)n_in;
    const long long F = end / h->H, gF = F / h->K;
    const long long done = gF * h->K + ((F - gF * h->K) / PSD_S) * PSD_S;  // last chunk boundary <= F
    const long long gid0 = psd_gid(h, h->done), gid1 = psd_gid(h, done);
    PsdSrc src;
    src.hist = h->d_hist[h->cur].p;
    src.in = in;
    src.hist_lo = h->hist_lo;
    src.in_lo = h->total;
    src.end = end;
    if (gid1 > gid0) {
        const long long row_base = h->done / h->K;
        const int rc = h->fused ? psd_run_fused(h, src, gid0, gid1, row_base, out, out_stride)
                                : psd_run_general(h, src, gid0, gid1, row_base, out, out_stride);
        if (rc) return rc;
        h->last_path = h->fused ? 2 : 1;
    }
    // carry the samples of the frames from `done` on: stream indices lo .. end - 1
    const long long lo = std::min(end, std::max(0LL, (done + 1) * h->H - h->N));
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
            SDR_CUDA_TRY(cudaMemcpyAsync((char *)dst.p + (size_t)from_old * es, (const char *)in + (size_t)(first_in - h->total) * es,
                                         (size_t)(end - first_in) * es, cudaMemcpyDeviceToDevice, st));
        h->cur ^= 1;
    }
    h->hist_lo = lo;
    h->total = end;
    h->done = done;
    return SDR_OK;
}

static int psd_check(const sdr_psd *h, const void *in, size_t n_in, const float *out, size_t out_cap, size_t out_stride,
                     size_t *n_spectra, size_t *ng) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_spectra) return SDR_ERR_BAD_DATA_PTR;
    *n_spectra = 0;
    if (n_in > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    *ng = sdr_psd_output_count(h, n_in);
    if (*ng > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (*ng > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (*ng > 0 && out_stride < (size_t)h->N) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_psd_process_dev(sdr_psd_t *h, const void *in, size_t n_in, float *out, size_t out_cap,
                                   size_t out_stride, size_t *n_spectra) {
    size_t ng = 0;
    int rc = psd_check(h, in, n_in, out, out_cap, out_stride, n_spectra, &ng);
    if (rc) return rc;
    if (((uintptr_t)in % psd_es(h)) != 0 || ((uintptr_t)out % 4) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = psd_run(h, in, n_in, out, out_stride);
    if (rc) return rc;
    *n_spectra = ng;
    return SDR_OK;
}

extern "C" int sdr_psd_process(sdr_psd_t *h, const void *in, size_t n_in, float *out, size_t out_cap, size_t out_stride,
                               size_t *n_spectra) {
    size_t ng = 0;
    int rc = psd_check(h, in, n_in, out, out_cap, out_stride, n_spectra, &ng);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t es = psd_es(h), N = (size_t)h->N;
    cudaStream_t st = h->stream.s;
    // chunks of about 32 MiB of input: H2D, compute, D2H in stream order
    const size_t chunk = std::max<size_t>(1, std::min(PSD_SLAB_BYTES / es, std::max<size_t>(n_in, 1)));
    const size_t rcap = chunk / (size_t)(h->H * h->K) + 1;  // spectra one chunk can complete
    rc = h->d_in.reserve(chunk * es);
    if (!rc) rc = h->d_out.reserve(rcap * N * sizeof(float));
    if (rc) return rc;
    size_t done_in = 0, done_out = 0;
    while (done_in < n_in) {
        const size_t cnt = std::min(chunk, n_in - done_in);
        const size_t cng = sdr_psd_output_count(h, cnt);
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_in.p, (const char *)in + done_in * es, cnt * es, cudaMemcpyHostToDevice, st));
        rc = psd_run(h, h->d_in.p, cnt, (float *)h->d_out.p, N);
        if (rc) return rc;
        if (cng > 0)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(out + done_out * out_stride, out_stride * sizeof(float), h->d_out.p,
                                           N * sizeof(float), N * sizeof(float), cng, cudaMemcpyDeviceToHost, st));
        done_in += cnt;
        done_out += cng;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_spectra = done_out;
    return SDR_OK;
}

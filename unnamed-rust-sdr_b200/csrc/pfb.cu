// pfb.cu -- sdr_pfb_*: polyphase filter bank.  One wideband stream -> M channels decimated by D.
// Channel k is Fir<Complex<f32>, Complex<f32>> with taps g_k[n] = h[n] e^{+2 pi i k n / M} (src/filter/fir.rs:23-32)
// followed by Decimate with wait D (src/signal/adapters/mod.rs:30-37):
//     y_k[m] = sum_{n<L} g_k[n] x[(m+1) D - 1 - n],   x[<0] = 0
// computed in polyphase form: branch p (taps h[t M + p]) gives
//     u_p[m] = sum_{t : t M + p < L} h[t M + p] x[(m+1) D - 1 - t M - p]        (one FMA chain, ascending t)
// stored at index (-p) mod M of frame m, and an unnormalised forward DFT of length M of that frame (the sdr_fft plan)
// gives y_0..y_{M-1}[m].  The work runs in slabs of frames whose c64 intermediate stays in L2: front end -> FFT
// (-> transpose to channel rows).
// Carried across calls: the last L - 1 inputs (raw format) and the stream position, so blocks of any size may be fed.
#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"

using namespace sdr;

namespace {

constexpr size_t PFB_SLAB_BYTES = (size_t)32 << 20;  // c64 intermediate per slab: two of them stay in the 126 MB L2
constexpr unsigned PFB_FLAGS = SDR_PFB_SHIFT | SDR_PFB_CHANNEL_MAJOR | SDR_PFB_GENERAL_KERNEL;
constexpr int PFB_REG_MAX = 32;  // (M / D) * T complex samples a thread may keep in registers

// Where the samples of one call live.  Stream index i is hist[i - hist_lo] for i < in_lo (the carried tail) and
// in[i - in_lo] for in_lo <= i < end; indices below lo (before the stream or before the carried tail) and at or past
// end read as zero -- only the register kernel's warm-up and padding ever asks for them, and never multiplies them.
struct PfbSrc {
    const void *hist;
    const void *in;
    long long lo, hist_lo, in_lo, end;
};

template <bool U8>
__device__ __forceinline__ float2 pfb_load(const PfbSrc &s, long long i) {
    if (i < s.lo || i >= s.end) return make_float2(0.f, 0.f);
    const bool h = i < s.in_lo;
    const void *base = h ? s.hist : s.in;
    const long long k = h ? i - s.hist_lo : i - s.in_lo;
    if (U8) return unpack_iq_u16(__ldg(reinterpret_cast<const uint16_t *>(base) + k));
    return __ldg(reinterpret_cast<const float2 *>(base) + k);
}

// taps of branch p: T_p = #{t : t M + p < L}
__device__ __forceinline__ int pfb_branch_taps(int p, int M, int L) { return p < L ? (L - 1 - p) / M + 1 : 0; }

// General front end: one thread per (branch p, frame).  Window samples come through L1 / L2.
template <bool U8>
__global__ void __launch_bounds__(256) pfb_front_general_kernel(PfbSrc src, const float *__restrict__ taps, int M,
                                                                 long long D, int L, long long j0, long long nf,
                                                                 float2 *__restrict__ u) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= M) return;
    const int Tp = pfb_branch_taps(p, M, L);
    const int col = p == 0 ? 0 : M - p;
    for (long long f = blockIdx.y; f < nf; f += gridDim.y) {
        const long long e = (j0 + f + 1) * D - 1 - p;
        float ar = 0.f, ai = 0.f;
        for (int t = 0; t < Tp; ++t) {
            const float hv = __ldg(taps + (size_t)t * M + p);
            const float2 x = pfb_load<U8>(src, e - (long long)t * M);
            ar = __fmaf_rn(hv, x.x, ar);
            ai = __fmaf_rn(hv, x.y, ai);
        }
        u[f * M + col] = make_float2(ar, ai);
    }
}

// Register-window front end for D | M, R = M / D, T <= TT, R * TT <= PFB_REG_MAX.  With q = m + 1, tap t of branch p
// reads x[(q - t R) D - 1 - p], so frame m only touches chain r = q mod R of the sequence s_p[q] = x[q D - 1 - p].
// Thread p keeps each chain's last TT values in registers; per frame it loads one sample (coalesced across p: the
// threads of a warp read consecutive samples) and runs the same FMA chain as the general kernel, so the bits agree.
// A thread covers the frames of `chunk` consecutive groups of R frames, after TT - 1 warm-up groups that only load.
template <bool U8, int R, int TT>
__global__ void __launch_bounds__(256, 2) pfb_front_reg_kernel(PfbSrc src, const float *__restrict__ taps, int M,
                                                               long long D, int L, long long j0, long long nf,
                                                               long long chunk, float2 *__restrict__ u) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= M) return;
    const int Tp = pfb_branch_taps(p, M, L);
    const int col = p == 0 ? 0 : M - p;
    float h[TT];
#pragma unroll
    for (int t = 0; t < TT; ++t) h[t] = t < Tp ? __ldg(taps + (size_t)t * M + p) : 0.f;
    float2 w[R][TT];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int t = 0; t < TT; ++t) w[r][t] = make_float2(0.f, 0.f);
    // groups g cover q = g R .. g R + R - 1; this slab's frames have q in [j0 + 1, j0 + nf]
    const long long g_first = (j0 + 1) / R, g_last = (j0 + nf) / R;
    const long long ga = g_first + (long long)blockIdx.y * chunk;
    if (ga > g_last) return;
    const long long gb = min(g_last, ga + chunk - 1);
    for (long long g = ga - (TT - 1); g <= gb; ++g) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const long long q = g * R + r;
            const float2 x = pfb_load<U8>(src, q * D - 1 - p);
#pragma unroll
            for (int t = TT - 1; t > 0; --t) w[r][t] = w[r][t - 1];
            w[r][0] = x;
            const long long f = q - 1 - j0;
            if (g >= ga && f >= 0 && f < nf) {
                float ar = 0.f, ai = 0.f;
#pragma unroll
                for (int t = 0; t < TT; ++t) {
                    if (t < Tp) {
                        ar = __fmaf_rn(h[t], w[r][t].x, ar);
                        ai = __fmaf_rn(h[t], w[r][t].y, ai);
                    }
                }
                u[f * M + col] = make_float2(ar, ai);
            }
        }
    }
}

// frames x M (contiguous) -> M rows of out_stride: out[k * out_stride + f] = y[f * M + k]
__global__ void pfb_transpose_kernel(const float2 *__restrict__ y, int M, long long nf, float2 *__restrict__ out,
                                     long long out_stride) {
    __shared__ float2 tile[32][33];
    const long long f0 = (long long)blockIdx.y * 32;
    const int k0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const long long f = f0 + i;
        const int k = k0 + threadIdx.x;
        if (f < nf && k < M) tile[i][threadIdx.x] = y[f * M + k];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int k = k0 + i;
        const long long f = f0 + threadIdx.x;
        if (f < nf && k < M) out[(long long)k * out_stride + f] = tile[threadIdx.x][i];
    }
}

// register-window geometry: R = M / D and the tap capacity TT, or false when the general kernel has to run
bool pfb_reg_geometry(size_t M, size_t D, size_t T, int *R, int *TT) {
    if (M % D != 0 || M / D > 8) return false;
    const int r = (int)(M / D);
    if (r & (r - 1)) return false;
    int tt = 4;
    while (tt < (int)T) tt *= 2;
    if (r * tt > PFB_REG_MAX) return false;
    *R = r;
    *TT = tt;
    return true;
}

template <bool U8, int R, int TT>
void pfb_launch_reg_t(const PfbSrc &s, const float *taps, int M, long long D, int L, long long j0, long long nf,
                      float2 *u, cudaStream_t st) {
    const int bd = std::min(256, (M + 31) / 32 * 32);
    const int gx = (M + bd - 1) / bd;
    // about two CTAs per SM per slab; every thread then pays TT - 1 warm-up groups for its chunk of groups
    const long long groups = (j0 + nf) / R - (j0 + 1) / R + 1;
    const long long want = std::max(1LL, (long long)(2 * current_sm_count()) / gx);
    long long chunk = std::max<long long>((groups + want - 1) / want, 2 * (TT - 1) / R + 1);
    chunk = std::max(chunk, (groups + 65534) / 65535);
    const unsigned gy = (unsigned)((groups + chunk - 1) / chunk);
    pfb_front_reg_kernel<U8, R, TT><<<dim3(gx, gy), bd, 0, st>>>(s, taps, M, D, L, j0, nf, chunk, u);
}

// every (R, TT) with R * TT <= PFB_REG_MAX that pfb_reg_geometry can return; false for any other pair
template <bool U8>
bool pfb_launch_reg(int R, int TT, const PfbSrc &s, const float *taps, int M, long long D, int L, long long j0,
                    long long nf, float2 *u, cudaStream_t st) {
#define PFB_REG_CASE(r, tt) \
    if (R == r && TT == tt) { pfb_launch_reg_t<U8, r, tt>(s, taps, M, D, L, j0, nf, u, st); return true; }
    PFB_REG_CASE(1, 4) PFB_REG_CASE(1, 8) PFB_REG_CASE(1, 16) PFB_REG_CASE(1, 32)
    PFB_REG_CASE(2, 4) PFB_REG_CASE(2, 8) PFB_REG_CASE(2, 16)
    PFB_REG_CASE(4, 4) PFB_REG_CASE(4, 8)
    PFB_REG_CASE(8, 4)
#undef PFB_REG_CASE
    return false;
}

}  // namespace

struct PfbHost {
    int dev = 0;
    size_t L = 0, M = 0, D = 1, T = 0, HL = 0;
    int fmt = SDR_FMT_C64;
    unsigned flags = 0;
    int reg_R = 0, reg_TT = 0;  // register-window geometry, 0 = general kernel
    std::vector<float> taps;    // T * M, zero padded
    long long total = 0;        // input samples seen; frames completed = total / D
};

static size_t pfb_es(const PfbHost *h) { return h->fmt == SDR_FMT_U8IQ ? 2 : 8; }

struct sdr_pfb : PfbHost {
    StreamRef stream;
    Owned<sdr_fft_t, sdr_fft_destroy> plan;
    DevBuf d_taps;
    DevBuf d_hist[2];           // the last HL inputs before `total`, raw format
    int cur = 0;
    DevBuf d_u, d_y, d_in, d_out;

    // taps, FFT plan and history buffers of a handle whose geometry fields are set
    int alloc(void *user_stream, const sdr_pfb *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_taps.upload(taps.data(), taps.size() * sizeof(float), stream.s))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(HL, 2) * pfb_es(this)))) return rc;
        sdr_fft_config_t fc;
        fc.n = M;
        fc.input_format = SDR_FMT_C64;
        fc.flags = (flags & SDR_PFB_SHIFT) ? SDR_FFT_SHIFT : 0u;
        fc.device = dev;
        fc.stream = (void *)stream.s;
        plan.reset(sdr_fft_create(&fc, &rc));
        if (!plan) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_pfb &src) {
        if (HL == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, HL * pfb_es(this), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_pfb_t *sdr_pfb_create(const sdr_pfb_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || cfg->n_taps == 0 || cfg->n_taps > ((size_t)1 << 24) || cfg->n_channels < 2 ||
        cfg->n_channels > 65536 || cfg->decimation == 0 || cfg->decimation > ((size_t)1 << 40) ||
        (cfg->input_format != SDR_FMT_U8IQ && cfg->input_format != SDR_FMT_C64) || (cfg->flags & ~PFB_FLAGS))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_pfb>(err, cfg->device, cfg->stream, [&](sdr_pfb &h) {
        h.L = cfg->n_taps;
        h.M = cfg->n_channels;
        h.D = cfg->decimation;
        h.T = (h.L + h.M - 1) / h.M;
        h.HL = h.L - 1;
        h.fmt = cfg->input_format;
        h.flags = cfg->flags;
        h.taps.assign(h.T * h.M, 0.0f);
        std::memcpy(h.taps.data(), cfg->taps, h.L * sizeof(float));
        if (!(h.flags & SDR_PFB_GENERAL_KERNEL) && !pfb_reg_geometry(h.M, h.D, h.T, &h.reg_R, &h.reg_TT))
            h.reg_R = h.reg_TT = 0;
        return SDR_OK;
    });
}

extern "C" void sdr_pfb_destroy(sdr_pfb_t *h) { destroy_handle(h); }

extern "C" int sdr_pfb_reset(sdr_pfb_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // indices below 0 read as zero, so the stale history is never used
    h->total = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_pfb_t *sdr_pfb_clone(const sdr_pfb_t *src, int *err) { return clone_handle<PfbHost>(src, err); }

// frames that the next n_in samples complete: frame j needs input sample (j + 1) * D - 1
extern "C" size_t sdr_pfb_output_count(const sdr_pfb_t *h, size_t n_in) {
    if (!h) return 0;
    const long long D = (long long)h->D;
    return (size_t)((h->total + (long long)n_in) / D - h->total / D);
}

// in: n_in device samples; out: nf frames, frame-major (row stride out_stride) or channel-major (M rows of out_stride)
static int pfb_run(sdr_pfb *h, const void *in, size_t n_in, float *out, size_t out_stride, size_t nf) {
    cudaStream_t st = h->stream.s;
    const size_t M = h->M, es = pfb_es(h);
    const long long D = (long long)h->D;
    const bool cmajor = (h->flags & SDR_PFB_CHANNEL_MAJOR) != 0;
    const float *taps = (const float *)h->d_taps.p;
    PfbSrc s;
    s.hist = h->d_hist[h->cur].p;
    s.in = in;
    s.in_lo = h->total;
    s.hist_lo = h->total - (long long)h->HL;
    s.lo = std::max(0LL, s.hist_lo);
    s.end = h->total + (long long)n_in;
    if (nf > 0) {
        const size_t slab = std::max<size_t>(1, std::min(nf, PFB_SLAB_BYTES / (M * 8)));
        int rc = h->d_u.reserve(slab * M * 8);
        if (rc) return rc;
        // frame-major output with stride M takes the FFT directly; any other layout goes through d_y
        const bool direct = !cmajor && out_stride == M && ((uintptr_t)out % 16) == 0 && (M * 8) % 16 == 0;
        if (!direct) {
            rc = h->d_y.reserve(slab * M * 8);
            if (rc) return rc;
        }
        const long long jbase = h->total / D;
        float2 *u = (float2 *)h->d_u.p;
        for (size_t f0 = 0; f0 < nf; f0 += slab) {
            const size_t cnt = std::min(slab, nf - f0);
            const long long j0 = jbase + (long long)f0;
            bool done = false;
            if (h->reg_R) {
                done = h->fmt == SDR_FMT_U8IQ
                           ? pfb_launch_reg<true>(h->reg_R, h->reg_TT, s, taps, (int)M, D, (int)h->L, j0, (long long)cnt, u, st)
                           : pfb_launch_reg<false>(h->reg_R, h->reg_TT, s, taps, (int)M, D, (int)h->L, j0, (long long)cnt, u, st);
            }
            if (!done) {
                dim3 grid((unsigned)((M + 255) / 256), (unsigned)std::min<size_t>(cnt, 65535));
                if (h->fmt == SDR_FMT_U8IQ)
                    pfb_front_general_kernel<true><<<grid, 256, 0, st>>>(s, taps, (int)M, D, (int)h->L, j0, (long long)cnt, u);
                else
                    pfb_front_general_kernel<false><<<grid, 256, 0, st>>>(s, taps, (int)M, D, (int)h->L, j0, (long long)cnt, u);
            }
            count_launch();
            rc = launch_status();
            if (rc) return rc;
            if (direct) {
                rc = sdr_fft_exec_dev(h->plan.get(), u, cnt, out + f0 * M * 2);
                if (rc) return rc;
                continue;
            }
            float2 *y = (float2 *)h->d_y.p;
            rc = sdr_fft_exec_dev(h->plan.get(), u, cnt, (float *)y);
            if (rc) return rc;
            if (cmajor) {
                pfb_transpose_kernel<<<dim3((unsigned)((M + 31) / 32), (unsigned)((cnt + 31) / 32)), dim3(32, 8), 0, st>>>(
                    y, (int)M, (long long)cnt, (float2 *)out + f0, (long long)out_stride);
                count_launch();
                rc = launch_status();
                if (rc) return rc;
            } else {
                SDR_CUDA_TRY(cudaMemcpy2DAsync(out + f0 * out_stride * 2, out_stride * 8, y, M * 8, M * 8, cnt,
                                               cudaMemcpyDeviceToDevice, st));
            }
        }
    }
    // history = the last HL samples of (history, input): keep the old tail that is still needed, then the input's tail
    if (h->HL > 0 && n_in > 0) {
        const size_t from_in = std::min(n_in, h->HL), from_old = h->HL - from_in;
        char *dst = (char *)h->d_hist[h->cur ^ 1].p;
        if (from_old > 0)
            SDR_CUDA_TRY(cudaMemcpyAsync(dst, (const char *)h->d_hist[h->cur].p + from_in * es, from_old * es,
                                         cudaMemcpyDeviceToDevice, st));
        SDR_CUDA_TRY(cudaMemcpyAsync(dst + from_old * es, (const char *)in + (n_in - from_in) * es, from_in * es,
                                     cudaMemcpyDeviceToDevice, st));
        h->cur ^= 1;
    }
    h->total += (long long)n_in;
    return SDR_OK;
}

static int pfb_check(const sdr_pfb *h, const void *in, size_t n_in, const float *out, size_t out_cap,
                     size_t out_stride, size_t *n_frames, size_t *nf) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_frames) return SDR_ERR_BAD_DATA_PTR;
    *n_frames = 0;
    if (n_in > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    *nf = sdr_pfb_output_count(h, n_in);
    if (*nf > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (*nf > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (*nf > 0 && out_stride < ((h->flags & SDR_PFB_CHANNEL_MAJOR) ? *nf : h->M)) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_pfb_process_dev(sdr_pfb_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                                   size_t out_stride, size_t *n_frames) {
    size_t nf = 0;
    int rc = pfb_check(h, in, n_in, out_c64, out_cap, out_stride, n_frames, &nf);
    if (rc) return rc;
    if (((uintptr_t)in % pfb_es(h)) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = pfb_run(h, in, n_in, out_c64, out_stride, nf);
    if (rc) return rc;
    *n_frames = nf;
    return SDR_OK;
}

extern "C" int sdr_pfb_process(sdr_pfb_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                               size_t out_stride, size_t *n_frames) {
    size_t nf = 0;
    int rc = pfb_check(h, in, n_in, out_c64, out_cap, out_stride, n_frames, &nf);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t M = h->M, es = pfb_es(h), D = h->D;
    const bool cmajor = (h->flags & SDR_PFB_CHANNEL_MAJOR) != 0;
    cudaStream_t st = h->stream.s;
    // chunks of at most ~32 MiB of input and about one slab of output frames: H2D, compute, D2H in stream order
    const size_t slab = std::max<size_t>(1, PFB_SLAB_BYTES / (M * 8));
    size_t chunk = std::max<size_t>(1, std::min(PFB_SLAB_BYTES / es, slab * D));
    chunk = std::min(chunk, std::max<size_t>(n_in, 1));
    const size_t fcap = chunk / D + 1;
    rc = h->d_in.reserve(chunk * es);
    if (!rc) rc = h->d_out.reserve(fcap * M * 8);
    if (rc) return rc;
    size_t done_in = 0, done_out = 0;
    while (done_in < n_in) {
        const size_t cnt = std::min(chunk, n_in - done_in);
        const size_t cnf = sdr_pfb_output_count(h, cnt);
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_in.p, (const char *)in + done_in * es, cnt * es, cudaMemcpyHostToDevice, st));
        rc = pfb_run(h, h->d_in.p, cnt, (float *)h->d_out.p, cmajor ? fcap : M, cnf);
        if (rc) return rc;
        if (cnf > 0) {
            if (cmajor)
                SDR_CUDA_TRY(cudaMemcpy2DAsync(out_c64 + done_out * 2, out_stride * 8, h->d_out.p, fcap * 8, cnf * 8, M,
                                               cudaMemcpyDeviceToHost, st));
            else
                SDR_CUDA_TRY(cudaMemcpy2DAsync(out_c64 + done_out * out_stride * 2, out_stride * 8, h->d_out.p, M * 8,
                                               M * 8, cnf, cudaMemcpyDeviceToHost, st));
        }
        done_in += cnt;
        done_out += cnf;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_frames = done_out;
    return SDR_OK;
}

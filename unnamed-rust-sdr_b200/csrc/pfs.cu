// pfs.cu -- sdr_pfs_*: polyphase synthesis filter bank.  M channel streams -> one stream at D times the frame rate;
// the transpose of sdr_pfb.  Channel k is zero-stuffed by D (sample m at index (m+1) D - 1), filtered by
// Fir<Complex<f32>, Complex<f32>> with taps f_k[n] = f[n] e^{+2 pi i k n / M} (src/filter/fir.rs:23-32), and summed:
//     xh[t] = sum_m sum_k f_k[t - (m+1) D + 1] y_k[m]
// Since sum_k y_k[m] e^{2 pi i k n / M} depends only on n mod M, this is V_m[r] = Y_m[(-r) mod M] with Y_m the
// unnormalised forward DFT of frame m (the sdr_fft plan), and
//     xh[t] = sum_{n < L, n = t+1 (mod D)} f[n] V_{(t+1-n)/D - 1}[n mod M]        (one FMA chain, ascending n)
// Write c = (t + 1) mod D and q = (t + 1 - c) / D, so t = q D + c - 1: output (c, q) takes tap n = c + i D from frame
// q - 1 - i, i < I_c = ceil((L - c) / D).  The work runs in slabs of frames whose c64 intermediate stays in L2:
// gather (layout flags, strides) -> FFT -> back end.
// Carried across calls: the transforms Y of the last H = ceil((L - 1) / D) frames and the stream position.
#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"

using namespace sdr;

namespace {

constexpr size_t PFS_SLAB_BYTES = (size_t)32 << 20;  // c64 intermediate per slab: two of them stay in the 126 MB L2
constexpr unsigned PFS_FLAGS = SDR_PFS_SHIFT | SDR_PFS_CHANNEL_MAJOR | SDR_PFS_GENERAL_KERNEL;
constexpr int PFS_REG_R_MAX = 8;    // M / D values a register-window thread loads per frame
constexpr int PFS_REG_TT_MAX = 32;  // accumulators (outputs in flight) a register-window thread keeps

// Where the transformed frames of one slab live.  Frame j (absolute) is hist[j - hist_lo] for j < y_lo (carried) and
// y[j - y_lo] for y_lo <= j < end; frames below lo (before the stream or before the carried ones) read as zero -- the
// definition's frames before the stream, and the register kernel's warm-up, which never multiplies them.
struct PfsSrc {
    const float2 *hist;
    const float2 *y;
    long long lo, hist_lo, y_lo, end;
};

// V_j[col] = Y_j[(-col) mod M]
__device__ __forceinline__ float2 pfs_load(const PfsSrc &s, long long j, int col, int M) {
    if (j < s.lo || j >= s.end) return make_float2(0.f, 0.f);
    const int b = col == 0 ? 0 : M - col;
    const float2 *p = j < s.y_lo ? s.hist + (j - s.hist_lo) * M : s.y + (j - s.y_lo) * M;
    return __ldg(p + b);
}

// taps of output phase c: I_c = #{i : c + i D < L}
__device__ __forceinline__ int pfs_phase_taps(long long c, long long D, int L) {
    return c < L ? (int)((L - 1 - c) / D) + 1 : 0;
}

// frame-major gather: u[f M + k] = in[f stride + src(k)], src(k) = (k + M/2) mod M with SHIFT (row i holds channel
// (i - M/2) mod M), else k.  A pure permutation.
__global__ void pfs_gather_frames_kernel(const float2 *__restrict__ in, long long stride, int M, long long nf,
                                         int shift, float2 *__restrict__ u) {
    const long long total = nf * M;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long f = e / M;
        const int k = (int)(e - f * M);
        const int src = shift ? (k + M / 2) % M : k;
        u[e] = in[f * stride + src];
    }
}

// channel-major gather (M rows of `stride`) -> frames x M, by 32 x 32 tiles: u[f M + k] = in[src(k) stride + f]
__global__ void pfs_gather_rows_kernel(const float2 *__restrict__ in, long long stride, int M, long long nf, int shift,
                                       float2 *__restrict__ u) {
    __shared__ float2 tile[32][33];
    const long long f0 = (long long)blockIdx.x * 32;
    const int k0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int k = k0 + i;
        const long long f = f0 + threadIdx.x;
        if (f < nf && k < M) {
            const int src = shift ? (k + M / 2) % M : k;
            tile[i][threadIdx.x] = in[(long long)src * stride + f];
        }
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const long long f = f0 + i;
        const int k = k0 + threadIdx.x;
        if (f < nf && k < M) u[f * M + k] = tile[threadIdx.x][i];
    }
}

// General back end: one thread per output t of the slab, t in [t0, t0 + nt).  V comes through L1 / L2.
__global__ void __launch_bounds__(256) pfs_back_general_kernel(PfsSrc src, const float *__restrict__ taps, int M,
                                                                long long D, int L, long long t0, long long nt,
                                                                float2 *__restrict__ out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nt; e += (long long)gridDim.x * blockDim.x) {
        const long long t = t0 + e;
        const long long c = (t + 1) % D, q = (t + 1) / D;
        const int Ic = pfs_phase_taps(c, D, L);
        float ar = 0.f, ai = 0.f;
        for (int i = 0; i < Ic; ++i) {
            const long long n = c + (long long)i * D;
            const float fv = __ldg(taps + n);
            const float2 v = pfs_load(src, q - 1 - i, (int)(n % M), M);
            ar = __fmaf_rn(fv, v.x, ar);
            ai = __fmaf_rn(fv, v.y, ai);
        }
        out[e] = make_float2(ar, ai);
    }
}

// Register-window back end for D | M, R = M / D, I_c <= TT.  Thread c owns output phase c in [0, D): outputs
// t = q D + c - 1.  Column n mod M of tap n = c + i D is c + (i mod R) D, so frame j is read at the R columns
// c + r D only, each exactly once (coalesced across c), and its value r feeds outputs q = j + 1 + i with i = r (mod R).
// The thread walks frames downwards: acc[i] holds output q = j + 1 + i, whose chain then has taps 0..i - 1, so the
// chain runs in ascending n like the general kernel's and the bits agree.  Output q leaves acc[TT - 1] complete after
// frame q - TT; a thread covers `chunk` outputs q after TT - 1 warm-up frames that complete none.
template <int R, int TT>
__global__ void __launch_bounds__(256, 1) pfs_back_reg_kernel(PfsSrc src, const float *__restrict__ taps, int M, int D,
                                                            int L, long long t0, long long nt, long long chunk,
                                                            float2 *__restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= D) return;
    const int Ic = pfs_phase_taps(c, D, L);
    float f[TT];
#pragma unroll
    for (int i = 0; i < TT; ++i) f[i] = i < Ic ? __ldg(taps + c + (size_t)i * D) : 0.f;
    // this phase's outputs in the slab: t = q D + c - 1 in [t0, t0 + nt)
    const long long q_first = (t0 + 1 - c + D - 1) / D, q_last = (t0 + nt - c) / D;
    const long long qa = q_first + (long long)blockIdx.y * chunk;
    if (qa > q_last) return;
    const long long qb = min(q_last, qa + chunk - 1);
    float2 acc[TT];
#pragma unroll
    for (int i = 0; i < TT; ++i) acc[i] = make_float2(0.f, 0.f);
#pragma unroll 1
    for (long long j = qb - 1; j >= qa - TT; --j) {
        float2 v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = pfs_load(src, j, c + r * D, M);
#pragma unroll
        for (int i = TT - 1; i > 0; --i) acc[i] = acc[i - 1];
        acc[0] = make_float2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < TT; ++i) {
            if (i < Ic) {
                acc[i].x = __fmaf_rn(f[i], v[i % R].x, acc[i].x);
                acc[i].y = __fmaf_rn(f[i], v[i % R].y, acc[i].y);
            }
        }
        const long long q = j + TT;
        if (q <= qb) out[q * D + c - 1 - t0] = acc[TT - 1];
    }
}

// register-window geometry: R = M / D and the accumulator count TT, or false when the general kernel has to run
bool pfs_reg_geometry(size_t M, size_t D, size_t L, int *R, int *TT) {
    if (M % D != 0 || M / D > (size_t)PFS_REG_R_MAX) return false;
    const int r = (int)(M / D);
    if (r & (r - 1)) return false;
    const size_t imax = (L + D - 1) / D;  // I_0, the most taps any phase has
    int tt = 8;
    while ((size_t)tt < imax) tt *= 2;
    if (tt > PFS_REG_TT_MAX) return false;
    *R = r;
    *TT = tt;
    return true;
}

template <int R, int TT>
void pfs_launch_reg_t(const PfsSrc &s, const float *taps, int M, int D, int L, long long t0, long long nt, float2 *out,
                      cudaStream_t st) {
    const int bd = std::min(256, (D + 31) / 32 * 32);
    const int gx = (D + bd - 1) / bd;
    // about two CTAs per SM per slab; every thread then pays TT - 1 warm-up frames for its chunk of outputs
    const long long outs = nt / D + 2;
    const long long want = std::max(1LL, (long long)(2 * current_sm_count()) / gx);
    long long chunk = std::max<long long>((outs + want - 1) / want, 2 * TT);
    chunk = std::max(chunk, (outs + 65534) / 65535);
    const unsigned gy = (unsigned)((outs + chunk - 1) / chunk);
    pfs_back_reg_kernel<R, TT><<<dim3(gx, gy), bd, 0, st>>>(s, taps, M, D, L, t0, nt, chunk, out);
}

// every (R, TT) that pfs_reg_geometry can return; false for any other pair
bool pfs_launch_reg(int R, int TT, const PfsSrc &s, const float *taps, int M, int D, int L, long long t0, long long nt,
                    float2 *out, cudaStream_t st) {
#define PFS_REG_CASE(r, tt) \
    if (R == r && TT == tt) { pfs_launch_reg_t<r, tt>(s, taps, M, D, L, t0, nt, out, st); return true; }
    PFS_REG_CASE(1, 8) PFS_REG_CASE(1, 16) PFS_REG_CASE(1, 32)
    PFS_REG_CASE(2, 8) PFS_REG_CASE(2, 16) PFS_REG_CASE(2, 32)
    PFS_REG_CASE(4, 8) PFS_REG_CASE(4, 16) PFS_REG_CASE(4, 32)
    PFS_REG_CASE(8, 8) PFS_REG_CASE(8, 16) PFS_REG_CASE(8, 32)
#undef PFS_REG_CASE
    return false;
}

}  // namespace

struct PfsHost {
    int dev = 0;
    size_t L = 0, M = 0, D = 1, H = 0;
    unsigned flags = 0;
    int reg_R = 0, reg_TT = 0;  // register-window geometry, 0 = general kernel
    std::vector<float> taps;
    long long total = 0;        // frames seen
};

struct sdr_pfs : PfsHost {
    StreamRef stream;
    Owned<sdr_fft_t, sdr_fft_destroy> plan;
    DevBuf d_taps;
    DevBuf d_hist[2];           // transforms of the H frames before `total`, frames x M
    int cur = 0;
    DevBuf d_u, d_y, d_in, d_out;

    // taps, FFT plan and history buffers of a handle whose geometry fields are set
    int alloc(void *user_stream, const sdr_pfs *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_taps.upload(taps.data(), taps.size() * sizeof(float), stream.s))) return rc;
        for (int i = 0; i < 2; ++i)
            if ((rc = d_hist[i].reserve(std::max<size_t>(H, 1) * M * 8))) return rc;
        sdr_fft_config_t fc;
        fc.n = M;
        fc.input_format = SDR_FMT_C64;
        fc.flags = 0;
        fc.device = dev;
        fc.stream = (void *)stream.s;
        plan.reset(sdr_fft_create(&fc, &rc));
        if (!plan) return rc;
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_pfs &src) {
        if (H == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, H * M * 8, cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_pfs_t *sdr_pfs_create(const sdr_pfs_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || cfg->n_taps == 0 || cfg->n_taps > ((size_t)1 << 24) || cfg->n_channels < 2 ||
        cfg->n_channels > 65536 || cfg->interpolation == 0 || cfg->interpolation > ((size_t)1 << 32) ||
        (cfg->flags & ~PFS_FLAGS))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_pfs>(err, cfg->device, cfg->stream, [&](sdr_pfs &h) {
        h.L = cfg->n_taps;
        h.M = cfg->n_channels;
        h.D = cfg->interpolation;
        h.H = (h.L - 1 + h.D - 1) / h.D;
        h.flags = cfg->flags;
        h.taps.assign(cfg->taps, cfg->taps + h.L);
        if (!(h.flags & SDR_PFS_GENERAL_KERNEL) && !pfs_reg_geometry(h.M, h.D, h.L, &h.reg_R, &h.reg_TT))
            h.reg_R = h.reg_TT = 0;
        return SDR_OK;
    });
}

extern "C" void sdr_pfs_destroy(sdr_pfs_t *h) { destroy_handle(h); }

extern "C" int sdr_pfs_reset(sdr_pfs_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // frames below 0 read as zero, so the stale history is never used
    h->total = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_pfs_t *sdr_pfs_clone(const sdr_pfs_t *src, int *err) { return clone_handle<PfsHost>(src, err); }

extern "C" size_t sdr_pfs_output_count(const sdr_pfs_t *h, size_t n_frames) {
    if (!h) return 0;
    return n_frames * h->D;
}

// in: nf device frames in the handle's layout with stride in_stride; out: nf * D samples
static int pfs_run(sdr_pfs *h, const float2 *in, size_t nf, size_t in_stride, float2 *out) {
    cudaStream_t st = h->stream.s;
    const size_t M = h->M, H = h->H;
    const long long D = (long long)h->D;
    const bool cmajor = (h->flags & SDR_PFS_CHANNEL_MAJOR) != 0;
    const int shift = (h->flags & SDR_PFS_SHIFT) ? 1 : 0;
    if (nf == 0) return SDR_OK;
    const size_t slab = std::max<size_t>(1, std::min(nf, PFS_SLAB_BYTES / (M * 8)));
    int rc = h->d_y.reserve(slab * M * 8);
    if (rc) return rc;
    float2 *y = (float2 *)h->d_y.p;
    for (size_t f0 = 0; f0 < nf; f0 += slab) {
        const size_t cnt = std::min(slab, nf - f0);
        const float2 *x = in + f0 * M;
        // frame-major, unshifted frames of stride M go to the FFT as they are; any other layout is gathered into d_u
        if (cmajor || shift || in_stride != M || ((uintptr_t)x % 16) != 0) {
            if ((rc = h->d_u.reserve(slab * M * 8))) return rc;
            float2 *u = (float2 *)h->d_u.p;
            if (cmajor)
                pfs_gather_rows_kernel<<<dim3((unsigned)((cnt + 31) / 32), (unsigned)((M + 31) / 32)), dim3(32, 8), 0, st>>>(
                    in + f0, (long long)in_stride, (int)M, (long long)cnt, shift, u);
            else
                pfs_gather_frames_kernel<<<(unsigned)std::min<size_t>((cnt * M + 255) / 256, 65535), 256, 0, st>>>(
                    in + f0 * in_stride, (long long)in_stride, (int)M, (long long)cnt, shift, u);
            count_launch();
            if ((rc = launch_status())) return rc;
            x = u;
        }
        if ((rc = sdr_fft_exec_dev(h->plan.get(), x, cnt, (float *)y))) return rc;
        PfsSrc s;
        s.hist = (const float2 *)h->d_hist[h->cur].p;
        s.y = y;
        s.y_lo = h->total;
        s.hist_lo = h->total - (long long)H;
        s.lo = std::max(0LL, s.hist_lo);
        s.end = h->total + (long long)cnt;
        const long long t0 = h->total * D, nt = (long long)cnt * D;
        float2 *o = out + f0 * (size_t)D;
        const float *taps = (const float *)h->d_taps.p;
        bool done = h->reg_R && pfs_launch_reg(h->reg_R, h->reg_TT, s, taps, (int)M, (int)D, (int)h->L, t0, nt, o, st);
        if (!done)
            pfs_back_general_kernel<<<(unsigned)std::min<long long>((nt + 255) / 256, 1 << 20), 256, 0, st>>>(
                s, taps, (int)M, D, (int)h->L, t0, nt, o);
        count_launch();
        if ((rc = launch_status())) return rc;
        // history = the transforms of the last H frames of (history, slab)
        if (H > 0) {
            const size_t from_y = std::min(cnt, H), from_old = H - from_y;
            char *dst = (char *)h->d_hist[h->cur ^ 1].p;
            if (from_old > 0)
                SDR_CUDA_TRY(cudaMemcpyAsync(dst, (const char *)h->d_hist[h->cur].p + from_y * M * 8, from_old * M * 8,
                                             cudaMemcpyDeviceToDevice, st));
            SDR_CUDA_TRY(cudaMemcpyAsync(dst + from_old * M * 8, y + (cnt - from_y) * M, from_y * M * 8,
                                         cudaMemcpyDeviceToDevice, st));
            h->cur ^= 1;
        }
        h->total += (long long)cnt;
    }
    return SDR_OK;
}

static int pfs_check(const sdr_pfs *h, const float *in, size_t n_frames, size_t in_stride, const float *out,
                     size_t out_cap, size_t *n_out) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    *n_out = 0;
    if (n_frames == 0) return SDR_OK;
    if (!in) return SDR_ERR_BAD_DATA_PTR;
    if (in_stride < ((h->flags & SDR_PFS_CHANNEL_MAJOR) ? n_frames : h->M)) return SDR_ERR_INVALID_ARG;
    if (sdr_pfs_output_count(h, n_frames) > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (!out) return SDR_ERR_BAD_DATA_PTR;
    return SDR_OK;
}

extern "C" int sdr_pfs_process_dev(sdr_pfs_t *h, const float *in_c64, size_t n_frames, size_t in_stride,
                                   float *out_c64, size_t out_cap, size_t *n_out) {
    int rc = pfs_check(h, in_c64, n_frames, in_stride, out_c64, out_cap, n_out);
    if (rc || n_frames == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = pfs_run(h, (const float2 *)in_c64, n_frames, in_stride, (float2 *)out_c64);
    if (rc) return rc;
    *n_out = n_frames * h->D;
    return SDR_OK;
}

extern "C" int sdr_pfs_process(sdr_pfs_t *h, const float *in_c64, size_t n_frames, size_t in_stride, float *out_c64,
                               size_t out_cap, size_t *n_out) {
    int rc = pfs_check(h, in_c64, n_frames, in_stride, out_c64, out_cap, n_out);
    if (rc || n_frames == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t M = h->M, D = h->D;
    const bool cmajor = (h->flags & SDR_PFS_CHANNEL_MAJOR) != 0;
    cudaStream_t st = h->stream.s;
    // chunks of about one slab of frames and at most ~32 MiB of output: H2D, compute, D2H in stream order
    size_t chunk = std::max<size_t>(1, std::min(PFS_SLAB_BYTES / (M * 8), PFS_SLAB_BYTES / (D * 8)));
    chunk = std::min(chunk, n_frames);
    rc = h->d_in.reserve(chunk * M * 8);
    if (!rc) rc = h->d_out.reserve(chunk * D * 8);
    if (rc) return rc;
    for (size_t done = 0; done < n_frames;) {
        const size_t cnt = std::min(chunk, n_frames - done);
        if (cmajor)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, cnt * 8, in_c64 + done * 2, in_stride * 8, cnt * 8, M,
                                           cudaMemcpyHostToDevice, st));
        else
            SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, M * 8, in_c64 + done * in_stride * 2, in_stride * 8, M * 8, cnt,
                                           cudaMemcpyHostToDevice, st));
        rc = pfs_run(h, (const float2 *)h->d_in.p, cnt, cmajor ? cnt : M, (float2 *)h->d_out.p);
        if (rc) return rc;
        SDR_CUDA_TRY(cudaMemcpyAsync(out_c64 + done * D * 2, h->d_out.p, cnt * D * 8, cudaMemcpyDeviceToHost, st));
        done += cnt;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_out = n_frames * D;
    return SDR_OK;
}

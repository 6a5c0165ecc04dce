// fft.cu -- K3: batched forward FFT, fused input unpack and fftshift + 1/sqrt(N) on store.
//
// Replaces rustfft's FFTplanner::plan_fft + process as called by fft::fft (src/fft.rs:10-12) and
// the shift/normalise loop of src/fft.rs:14-26 (and rfft's drain, src/fft.rs:34-36).
//
// Algorithm: Stockham autosort, decimation in time, radix-16 passes held in registers (a final
// radix 2/4/8 pass when log2 N is not a multiple of 4).  Every thread owns 16 points; pass data is
// exchanged through padded shared memory (index a -> a + a/16, which makes both the stride-16
// scatter of the first pass and the unit-stride gathers of later passes bank-conflict free).
// Twiddles come from a table computed on the host in f64 and rounded to f32 (as rustfft does).
//
//   n = 16 .. 16384    one kernel; a CTA holds whole transforms in shared memory (one HBM pass)
//   n = 32768, 65536   two kernels (four-step): 256-point column FFTs, then (n/256)-point column
//                      FFTs with the W_n^{k r} twiddle folded into the load.  The intermediate is
//                      written in place in the output buffer.
#include <cstdlib>

#include "kernels.h"
#include "fft_core.cuh"
#include "ptx.cuh"

namespace sdr {

namespace {

__device__ __forceinline__ int pad(int a) { return a + (a >> 4); }
__host__ __device__ constexpr int padlen(int n) { return n + (n >> 4) + 1; }

// One Stockham pass over a length-L sequence resident in shared memory.  TC = L/16 threads
// cooperate; thread t owns butterflies i = t + vi*TC (vi < 16/R), whose s-th input is element
// t + (vi + s*(16/R))*TC -- i.e. register e always maps to element t + e*TC.
template <int LOGL, int R, int PLOG>
__device__ __forceinline__ void fft_pass(float2 *s, int t, const float2 *__restrict__ tw, int tw_stride) {
    constexpr int L = 1 << LOGL, TC = L / 16, NB = 16 / R, p = 1 << PLOG;
    float2 v[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = s[pad(t + e * TC)];
    if (PLOG > 0) {
        constexpr int tstep = L / (p * R);
#pragma unroll
        for (int vi = 0; vi < NB; ++vi) {
            const int k = (t + vi * TC) & (p - 1);
#pragma unroll
            for (int q = 1; q < R; ++q) {
                const float2 w = __ldg(tw + (long long)(q * k * tstep) * tw_stride);
                v[vi + q * NB] = cmul(v[vi + q * NB], w);
            }
        }
    }
#pragma unroll
    for (int vi = 0; vi < NB; ++vi) dft<R, NB>(v + vi);
    __syncthreads();
#pragma unroll
    for (int vi = 0; vi < NB; ++vi) {
        const int i = t + vi * TC;
        const int k = i & (p - 1);
        const int base = (i - k) * R + k;
#pragma unroll
        for (int q = 0; q < R; ++q) s[pad(base + q * p)] = v[vi + q * NB];
    }
    __syncthreads();
}

// all passes: radix 16 while 4 bits remain, then one pass of radix 2^(LOGL % 4)
template <int LOGL, int PLOG>
__device__ __forceinline__ void fft_core(float2 *s, int t, const float2 *__restrict__ tw, int tw_stride) {
    if constexpr (PLOG < LOGL) {
        constexpr int rem = LOGL - PLOG;
        constexpr int RL = rem >= 4 ? 4 : rem;
        fft_pass<LOGL, (1 << RL), PLOG>(s, t, tw, tw_stride);
        fft_core<LOGL, PLOG + RL>(s, t, tw, tw_stride);
    }
}

template <int FMT>
__device__ __forceinline__ float2 load_elem(const void *in, long long idx) {
    if (FMT == SDR_FMT_U8IQ) return unpack_iq_u16(__ldg(reinterpret_cast<const uint16_t *>(in) + idx));
    if (FMT == SDR_FMT_C64) return __ldg(reinterpret_cast<const float2 *>(in) + idx);
    return make_float2(__ldg(reinterpret_cast<const float *>(in) + idx), 0.0f);
}

// where spectrum bin k lands in the output row, or -1 if dropped (rfft)
__device__ __forceinline__ int out_slot(int k, int n, unsigned flags) {
    if (flags & SDR_FFT_RFFT) return (k < n - n / 2) ? k : -1;
    if (flags & SDR_FFT_SHIFT) return (k + n / 2) & (n - 1);
    return k;
}

// ---- n <= 16384: whole transforms per CTA ------------------------------------------------
template <int LOGN, int FMT>
__global__ void __launch_bounds__((1 << LOGN) / 16 > 256 ? (1 << LOGN) / 16 : 256)
fft_cta_kernel(FftArgs a) {
    constexpr int N = 1 << LOGN, TC = N / 16;
    constexpr int THREADS = TC > 256 ? TC : 256;
    constexpr int SEQ = THREADS / TC;
    constexpr int SSTRIDE = padlen(N);
    extern __shared__ float4 smem4[];
    float2 *sm = reinterpret_cast<float2 *>(smem4);
    const int tid = threadIdx.x;
    const long long seq0 = (long long)blockIdx.x * SEQ;
    const int nseq = (int)min((long long)SEQ, a.batches - seq0);
    const int out_len = (a.flags & SDR_FFT_RFFT) ? N - N / 2 : N;

    for (int idx = tid; idx < SEQ * N; idx += THREADS) {
        const int q = idx >> LOGN, j = idx & (N - 1);
        float2 v = make_float2(0.0f, 0.0f);
        if (q < nseq) v = load_elem<FMT>(a.in, (seq0 + q) * N + j);
        sm[q * SSTRIDE + pad(j)] = v;
    }
    __syncthreads();
    fft_core<LOGN, 0>(sm + (tid / TC) * SSTRIDE, tid % TC, a.tw, 1);
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    for (int idx = tid; idx < SEQ * N; idx += THREADS) {
        const int q = idx >> LOGN, j = idx & (N - 1);  // j = output slot
        if (q >= nseq || j >= out_len) continue;
        int k = j;
        if (!(a.flags & SDR_FFT_RFFT) && (a.flags & SDR_FFT_SHIFT)) k = (j + N / 2) & (N - 1);  // src bin
        float2 v = sm[q * SSTRIDE + pad(k)];
        if (norm) { v.x *= a.norm; v.y *= a.norm; }
        a.out[(seq0 + q) * out_len + j] = v;
    }
}

// ---- n = 1024, the headline size: one warp per transform, 32 points per lane -----------------
// 1024 = 32 x 32: two radix-32 passes held entirely in registers and ONE exchange through
// warp-private shared memory, so the only synchronisation is __syncwarp().  Persistent warps loop
// over transforms; for u8 IQ the next transform's 2 KB of bytes is prefetched with cp.async while
// the current one is computed, so HBM latency is hidden with only 16 warps per SM.  The pass-2
// twiddles W_1024^{q*lane} live in a [31][32] shared table built once per CTA from the host f64
// table (exact values, conflict-free reads).  When 1/sqrt(N) is a power of two (N = 4^k) the
// normalisation is folded into the unpack constants (u8) or the twiddle table (c64): scaling by a
// power of two commutes with every rounding, so the result is bit-identical to scaling afterwards.

constexpr int W1K_WARPS = 8;  // 8 warps share one twiddle table; 2 CTAs (16 warps, ~214 KB smem) per SM
constexpr int W1K_XCH = 33 * 32;  // padded exchange, float2 per warp
__host__ __device__ constexpr size_t w1k_smem(int fmt) {
    return (size_t)(31 * 32 + W1K_WARPS * W1K_XCH) * sizeof(float2) + (fmt == SDR_FMT_U8IQ ? W1K_WARPS * 4096 : 0);
}

// SHIFT: 0 / 1 = fftshift off / on at compile time (u8 input: the 32 output addresses of a lane become immediates,
// +2.5 %), 2 = read from the flags at run time (c64 input, where the specialised code measured 7 % slower)
// TMA (u8 input): the next transform's 2 KB arrive by ONE cp.async.bulk (UBLKCP) issued by lane 0 and completing on a
// per-(warp, buffer) mbarrier, instead of four LDGSTS per lane and a wait_group: the same bytes over the same path into
// shared memory, 128 fewer issued instructions per transform in an issue-bound kernel.  TMA = false keeps the cp.async
// loader (A/B switch SDR_FFT_NO_TMA=1).
template <int FMT, int SHIFT, bool TMA = false>
__global__ void __launch_bounds__(W1K_WARPS * 32, 2) fft1024_warp_kernel(FftArgs a) {
    constexpr int N = 1024;
    extern __shared__ float4 smem4[];
    __shared__ __align__(8) uint64_t tma_bar[W1K_WARPS][2];
    float2 *tw_s = reinterpret_cast<float2 *>(smem4);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float2 *xch = tw_s + 31 * 32 + warp * W1K_XCH;
    unsigned char *raw = reinterpret_cast<unsigned char *>(tw_s + 31 * 32 + W1K_WARPS * W1K_XCH) + warp * 4096;
    const bool shift = SHIFT == 2 ? (a.flags & SDR_FFT_SHIFT) != 0 : SHIFT == 1;
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    const float fold = norm ? a.norm : 1.0f;  // 1/32: exact power of two
    for (int idx = tid; idx < 31 * 32; idx += W1K_WARPS * 32) {
        const int q = idx / 32 + 1, l = idx % 32;
        float2 t = __ldg(a.tw + q * l);
        if (FMT != SDR_FMT_U8IQ) { t.x *= fold; t.y *= fold; }
        tw_s[idx] = t;
    }
    __syncthreads();
    const long long nwarps = (long long)gridDim.x * W1K_WARPS;
    long long b = (long long)blockIdx.x * W1K_WARPS + warp;
    const float us = 0.0078125f * fold, uo = -65537.0f * fold;
    const unsigned char *in8 = reinterpret_cast<const unsigned char *>(a.in);
    int buf = 0;
    uint32_t tph = 0;  // bit i = parity of buffer i's mbarrier
    const uint32_t bar_s = smem_u32(&tma_bar[warp][0]), raw_s = smem_u32(raw);
    auto tma_load = [&](long long bb, int bf) {  // lane 0 only
        mbar_arrive_expect_tx(bar_s + 8u * bf, 2048);
        tma_bulk_g2s(raw_s + 2048u * bf, in8 + bb * 2048, 2048, bar_s + 8u * bf);
    };
    if (FMT == SDR_FMT_U8IQ && TMA) {
        if (lane == 0) {
            mbar_init(bar_s, 1);
            mbar_init(bar_s + 8u, 1);
            mbar_init_fence();
            if (b < a.batches) tma_load(b, 0);
        }
        __syncwarp();
    } else if (FMT == SDR_FMT_U8IQ && b < a.batches) {
#pragma unroll
        for (int i = 0; i < 4; ++i) cp_async16(raw + (i * 32 + lane) * 16, in8 + b * 2048 + (i * 32 + lane) * 16);
        cp_async_commit();
    }
    for (; b < a.batches; b += nwarps) {
        float2 v[32], w[32];
        if (FMT == SDR_FMT_U8IQ) {
            const long long nb = b + nwarps;
            if (TMA) {
                // buffer buf ^ 1 was last read one iteration ago, before that iteration's closing __syncwarp
                if (lane == 0 && nb < a.batches) tma_load(nb, buf ^ 1);
                mbar_wait(bar_s + 8u * buf, (tph >> buf) & 1u);
                tph ^= 1u << buf;
            } else if (nb < a.batches) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    cp_async16(raw + (buf ^ 1) * 2048 + (i * 32 + lane) * 16, in8 + nb * 2048 + (i * 32 + lane) * 16);
                cp_async_commit();
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncwarp();
            const unsigned short *r16 = reinterpret_cast<const unsigned short *>(raw + buf * 2048);
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const unsigned h = r16[lane + 32 * e];
                const unsigned mi = __byte_perm(h, 0x4B000000u, 0x7540u), mq = __byte_perm(h, 0x4B000000u, 0x7541u);
                v[e] = make_float2(__fmaf_rn(__uint_as_float(mi), us, uo), __fmaf_rn(__uint_as_float(mq), us, uo));
            }
            buf ^= 1;
        } else {
            const float2 *src = reinterpret_cast<const float2 *>(a.in) + b * N + lane;
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = __ldg(src + 32 * e);
        }
        dft32<FMT == SDR_FMT_U8IQ>(v, w);  // packed complex adds: +4 % for u8 input, -8 % for c64 (measured)
#pragma unroll
        for (int s = 0; s < 32; ++s) xch[33 * lane + s] = w[s];
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = xch[lane + 33 * e];
#pragma unroll
        for (int q = 1; q < 32; ++q) v[q] = cmul(v[q], tw_s[(q - 1) * 32 + lane]);
        if (FMT != SDR_FMT_U8IQ && norm) { v[0].x *= fold; v[0].y *= fold; }
        dft32<FMT == SDR_FMT_U8IQ>(v, w);
        float2 *dst = a.out + b * N + lane;
#pragma unroll
        for (int s = 0; s < 32; ++s) dst[32 * (shift ? (s ^ 16) : s)] = w[s];
        __syncwarp();
    }
}

template <int FMT>
int launch_w1k(const FftArgs &a, cudaStream_t st) {
    const size_t smem = w1k_smem(FMT);
    const bool shift = (a.flags & SDR_FFT_SHIFT) != 0;
    static const bool no_tma = std::getenv("SDR_FFT_NO_TMA") != nullptr;  // A/B switch (tuning)
    auto kern = FMT != SDR_FMT_U8IQ ? fft1024_warp_kernel<FMT, 2, false>
                : no_tma ? (shift ? fft1024_warp_kernel<FMT, 1, false> : fft1024_warp_kernel<FMT, 0, false>)
                         : (shift ? fft1024_warp_kernel<FMT, 1, true> : fft1024_warp_kernel<FMT, 0, true>);
    const int sms = current_sm_count();
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    long long ctas = (a.batches + W1K_WARPS - 1) / W1K_WARPS;
    if (ctas > (long long)sms * 2) ctas = (long long)sms * 2;
    kern<<<(unsigned)ctas, W1K_WARPS * 32, smem, st>>>(a);
    count_launch();
    return launch_status();
}

// ---- n = 256 .. 8192 (other than 1024): persistent CTA, registers + one shared exchange per pass ------------
// Same Stockham passes as fft_cta_kernel, without its staging round trips: the first pass loads straight from
// global memory into registers (element t + e*TC: coalesced), the last pass stores straight from registers, middle
// passes exchange through padded shared memory.  Twiddles never touch global memory in the loop: middle passes read
// per-pass shared tables [q][k] (conflict free), the last pass keeps its (R-1)*16/R per-thread twiddles in
// registers (a thread sees the same k for every transform because the CTA is persistent).  Threads of one
// transform synchronise with a named barrier (or __syncwarp when a transform fits in a warp), so the transforms
// sharing a CTA drift freely.
template <int TC>
__device__ __forceinline__ void group_sync(int group) {
    if (TC <= 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(TC));
}

template <int LOGN>
struct Reg2Plan {
    static constexpr int N = 1 << LOGN, TC = N / 16;
    static constexpr int THREADS = TC > 256 ? TC : 256;
    static constexpr int SEQ = THREADS / TC;
    static constexpr int NP = (LOGN + 3) / 4;                 // passes
    // FADD2 / packed complex adds (common.cuh): measured per size on one box, +3 % at 256 and 4096, -4 % at 8192
    static constexpr bool PACKED = LOGN != 13;
    static constexpr int RLAST = 1 << (LOGN - 4 * (NP - 1));  // radix of the last pass (16 if LOGN % 4 == 0)
    static constexpr int NBLAST = 16 / RLAST;
    // shared twiddle tables of the middle passes (pass j, 1 <= j <= NP-2): 15 * 16^j entries each
    __host__ __device__ static constexpr int tab_entries() {
        int e = 0, p = 16;
        for (int j = 1; j <= NP - 2; ++j) { e += 15 * p; p *= 16; }
        return e;
    }
    // one transform per CTA: the NEXT transform's input is prefetched (cp.async) into a raw buffer while this one is
    // computed, so a lone CTA per SM (n = 8192) still overlaps its HBM reads with its arithmetic
    static constexpr bool PREFETCH = (SEQ == 1) && (LOGN >= 13);  // measured: +4 % at 8192, -5 % at 4096 (2 CTAs per SM already overlap)
    __host__ __device__ static constexpr size_t raw_offset() { return (((size_t)SEQ * padlen(N) + tab_entries()) * sizeof(float2) + 15) / 16 * 16; }
    __host__ __device__ static constexpr size_t smem_bytes(int elem_bytes) { return raw_offset() + (PREFETCH ? (size_t)N * elem_bytes : 0); }
};
template <int FMT> struct FmtBytes { static constexpr int v = FMT == SDR_FMT_U8IQ ? 2 : FMT == SDR_FMT_C64 ? 8 : 4; };
template <int FMT>
__device__ __forceinline__ float2 raw_elem(const unsigned char *raw, int idx) {
    if (FMT == SDR_FMT_U8IQ) return unpack_iq_u16(*reinterpret_cast<const uint16_t *>(raw + 2 * idx));
    if (FMT == SDR_FMT_C64) return *reinterpret_cast<const float2 *>(raw + 8 * idx);
    return make_float2(*reinterpret_cast<const float *>(raw + 4 * idx), 0.0f);
}

// middle pass j (sub-size p = 16^j, radix 16): shared -> registers -> shared
template <int LOGN, int PLOG>
__device__ __forceinline__ void reg2_middle(float2 *sx, const float2 *tab, int t, int group) {
    constexpr bool PK = Reg2Plan<LOGN>::PACKED;
    constexpr int N = 1 << LOGN, TC = N / 16, p = 1 << PLOG;
    // pad(a + c) = pad(a) + c + c/16 when c is a multiple of 16 (no carry out of the low nibble): one pad() per pass,
    // the 16 elements at immediate offsets (the per-element shifts were a fifth of this kernel's issue slots)
    static_assert(TC % 16 == 0 && p % 16 == 0, "padded offsets");
    float2 v[16];
    const float2 *ld = sx + pad(t);
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = ld[e * (TC + TC / 16)];
    const int k = t & (p - 1);
#pragma unroll
    for (int q = 1; q < 16; ++q) v[q] = cmul(v[q], tab[(q - 1) * p + k]);
    dft<16, 1, PK>(v);
    group_sync<TC>(group);
    const int base = (t - k) * 16 + k;
    float2 *stp = sx + pad(base);
#pragma unroll
    for (int q = 0; q < 16; ++q) stp[q * (p + p / 16)] = v[q];
    group_sync<TC>(group);
}

// REGPF (n = 2048 .. 8192, c64): the next transform's pass-0 inputs are prefetched into REGISTERS (16 LDG.64 per thread, issued
// behind pass 0, consumed one transform later) instead of a cp.async raw copy in shared memory: the raw copy cost 128 KB
// of the 512 KB of shared-memory traffic per transform in a kernel whose phases are serialised by CTA-wide barriers.
template <int LOGN, int FMT, bool REGPF = false>
__global__ void __launch_bounds__(Reg2Plan<LOGN>::THREADS, (Reg2Plan<LOGN>::THREADS <= 256) ? 2 : 1)
fft_reg2_kernel(FftArgs a) {
    using PL = Reg2Plan<LOGN>;
    constexpr int N = PL::N, TC = PL::TC, THREADS = PL::THREADS, SEQ = PL::SEQ, NP = PL::NP;
    constexpr int RL = PL::RLAST, NBL = PL::NBLAST;
    extern __shared__ float4 smem4[];
    float2 *sm = reinterpret_cast<float2 *>(smem4);
    float2 *tabs = sm + SEQ * padlen(N);
    const int tid = threadIdx.x, group = tid / TC, t = tid % TC;
    float2 *sx = sm + group * padlen(N);

    // middle-pass tables: tab_j[(q-1)*p + k] = W_{16p}^{q k} = W_N^{q k N/(16p)}
    {
        int off = 0, p = 16;
#pragma unroll
        for (int j = 1; j <= NP - 2; ++j) {
            for (int idx = tid; idx < 15 * p; idx += THREADS) {
                const int q = idx / p + 1, k = idx % p;
                tabs[off + idx] = __ldg(a.tw + (long long)q * k * (N / (16 * p)));
            }
            off += 15 * p;
            p *= 16;
        }
    }
    // last-pass twiddles of this thread: butterfly vi has k = t + vi*TC, element q gets W_N^{q k}
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    float2 twl[NBL][RL - 1];
#pragma unroll
    for (int vi = 0; vi < NBL; ++vi)
#pragma unroll
        for (int q = 1; q < RL; ++q) twl[vi][q - 1] = __ldg(a.tw + (long long)q * (t + vi * TC));
    __syncthreads();

    const bool shift = (a.flags & SDR_FFT_SHIFT) != 0 && !(a.flags & SDR_FFT_RFFT);
    const int out_len = (a.flags & SDR_FFT_RFFT) ? N - N / 2 : N;
    constexpr bool PF = PL::PREFETCH && !REGPF;
    constexpr int ES = FmtBytes<FMT>::v;
    float2 nx[REGPF ? 16 : 1];
    if (REGPF && (long long)blockIdx.x * SEQ + group < a.batches) {
#pragma unroll
        for (int e = 0; e < 16; ++e) nx[REGPF ? e : 0] = load_elem<FMT>(a.in, ((long long)blockIdx.x * SEQ + group) * N + t + e * TC);
    }
    unsigned char *raw = reinterpret_cast<unsigned char *>(smem4) + PL::raw_offset();
    auto issue_raw = [&](long long b) {
        const unsigned char *src = reinterpret_cast<const unsigned char *>(a.in) + b * N * ES;
#pragma unroll
        for (int i = 0; i < (N * ES / 16 + THREADS - 1) / THREADS; ++i) {
            const int q = tid + THREADS * i;
            if (q < N * ES / 16) cp_async16(raw + 16 * q, src + 16 * q);
        }
        cp_async_commit();
    };
    if (PF && (long long)blockIdx.x < a.batches) issue_raw(blockIdx.x);
    for (long long b0 = (long long)blockIdx.x * SEQ; b0 < a.batches; b0 += (long long)gridDim.x * SEQ) {
        const long long b = b0 + group;
        const bool live = b < a.batches;
        float2 v[16];
        // ---- pass 0: global (or the prefetched raw copy) -> registers, radix 16, no twiddles ----
        if (PF) {
            cp_async_wait<0>();
            __syncthreads();
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = raw_elem<FMT>(raw, t + e * TC);
            __syncthreads();  // the raw buffer is free: fetch the next transform behind this one's arithmetic
            if (b0 + gridDim.x < a.batches) issue_raw(b0 + gridDim.x);
        } else if (REGPF) {
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = nx[REGPF ? e : 0];
            const long long nb = b + (long long)gridDim.x * SEQ;
            if (nb < a.batches) {
#pragma unroll
                for (int e = 0; e < 16; ++e) nx[REGPF ? e : 0] = load_elem<FMT>(a.in, nb * N + t + e * TC);
            }
        } else {
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = live ? load_elem<FMT>(a.in, b * N + t + e * TC) : make_float2(0.f, 0.f);
        }
        dft<16, 1, PL::PACKED>(v);
        if (NP == 1) {
            // (N == 16 is not dispatched here)
        }
        {
            float2 *st0 = sx + 17 * t;  // pad(16 t + q) = 17 t + q for q < 16
#pragma unroll
            for (int q = 0; q < 16; ++q) st0[q] = v[q];
        }
        group_sync<TC>(group);
        // ---- middle passes ----
        if (NP >= 3) reg2_middle<LOGN, 4>(sx, tabs, t, group);
        if (NP >= 4) reg2_middle<LOGN, 8>(sx, tabs + 15 * 16, t, group);
        // ---- last pass: shared -> registers, per-thread twiddles, registers -> global ----
        {
            const float2 *ld = sx + pad(t);  // pad(t + e TC) = pad(t) + e (TC + TC/16), TC a multiple of 16
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = ld[e * (TC + TC / 16)];
        }
#pragma unroll
        for (int vi = 0; vi < NBL; ++vi)
#pragma unroll
            for (int q = 1; q < RL; ++q) v[vi + q * NBL] = cmul(v[vi + q * NBL], twl[vi][q - 1]);
#pragma unroll
        for (int vi = 0; vi < NBL; ++vi) dft<RL, NBL, PL::PACKED>(v + vi);
        if (live) {
            float2 *dst = a.out + b * out_len;
#pragma unroll
            for (int e = 0; e < 16; ++e) {
                // register e = vi + q*NBL holds bin (t + vi*TC) + q*(N/RL) = t + e*TC
                int k = t + e * TC;
                if (shift) k = (k + N / 2) & (N - 1);
                float2 o = v[e];
                if (norm) { o.x *= a.norm; o.y *= a.norm; }
                if (k < out_len) dst[k] = o;
            }
        }
        group_sync<TC>(group);  // the exchange buffer is rewritten by the next transform
    }
}

template <int LOGN, int FMT>
int launch_cta(const FftArgs &a, cudaStream_t st);

template <int LOGN, int FMT>
int launch_reg2(const FftArgs &a, cudaStream_t st) {
    using PL = Reg2Plan<LOGN>;
    static const int mode8k = std::getenv("SDR_FFT8K") ? std::atoi(std::getenv("SDR_FFT8K")) : 1;  // A/B switch: 0 = cp.async raw copy
    // register prefetch below 8192: measured on one box (profiles/r02_ab_fft_regpf.txt) +7-9 % at 2048 and 4096 (two CTAs
    // per SM, 117-122 registers), -4 % / -9 % at 256 / 512.  A/B switch SDR_FFT_REGPF_MIN = smallest log2 n that uses it.
    static const int regpf_min = std::getenv("SDR_FFT_REGPF_MIN") ? std::atoi(std::getenv("SDR_FFT_REGPF_MIN")) : 11;
    constexpr bool CAN_REGPF = (PL::PREFETCH || LOGN >= 11) && FMT == SDR_FMT_C64;
    const bool regpf = CAN_REGPF && (PL::PREFETCH ? mode8k == 1 : LOGN >= regpf_min);
    const size_t smem = regpf ? PL::raw_offset() : PL::smem_bytes(FmtBytes<FMT>::v);
    if (!regpf && PL::PREFETCH && (((uintptr_t)a.in) & 15)) return launch_cta<LOGN, FMT>(a, st);  // cp.async needs 16-byte rows
    void (*kern)(FftArgs) = fft_reg2_kernel<LOGN, FMT, false>;
    if constexpr (CAN_REGPF) { if (regpf) kern = fft_reg2_kernel<LOGN, FMT, true>; }
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int sms = current_sm_count();
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, PL::THREADS, smem);
    if (per_sm < 1) per_sm = 1;
    long long ctas = (a.batches + PL::SEQ - 1) / PL::SEQ;
    if (ctas > (long long)sms * per_sm) ctas = (long long)sms * per_sm;
    kern<<<(unsigned)ctas, PL::THREADS, smem, st>>>(a);
    count_launch();
    return launch_status();
}

// ---- n = 2^15, 2^16: four-step, tile of 16 columns per CTA --------------------------------
// STEP 0: view x as [256][M] (M = n/256); 256-point FFT down each column c; result row-major
//         scratch[256*c + k2] (in the output buffer).
// STEP 1: view scratch as [M][256]; element r of column k is scratch[k + 256 r] * W_n^{k r};
//         M-point FFT down the column; bin k1 is X[k + 256 k1].
template <int LOGL, int FMT, int STEP>
__global__ void __launch_bounds__(16 * ((1 << LOGL) / 16)) fft_cols_kernel(FftArgs a) {
    constexpr int L = 1 << LOGL, TC = L / 16, THREADS = 16 * TC;
    constexpr int SSTRIDE = padlen(L);  // odd multiple-of-2 offset keeps the 16 columns on distinct banks
    extern __shared__ float4 smem4[];
    float2 *sm = reinterpret_cast<float2 *>(smem4);
    const int tid = threadIdx.x;
    const int n = 1 << a.log_n;
    const int M = n >> 8;
    const int ncol_tiles = (STEP == 0 ? M : 256) / 16;
    const long long b = blockIdx.x / ncol_tiles;
    const int col0 = (blockIdx.x % ncol_tiles) * 16;
    const int cstride = (STEP == 0) ? M : 256;  // distance between consecutive rows of a column
    const int c = tid & 15;
    float2 *xb = a.out + b * n;  // scratch / output row of this transform (n complex)
    for (int r = tid >> 4; r < L; r += THREADS / 16) {
        float2 v;
        if (STEP == 0) {
            v = load_elem<FMT>(a.in, b * n + (long long)(col0 + c) + (long long)cstride * r);
        } else {
            v = xb[(col0 + c) + cstride * r];
            v = cmul(v, __ldg(a.tw + (long long)(col0 + c) * r));
        }
        sm[c * SSTRIDE + pad(r)] = v;
    }
    __syncthreads();
    fft_core<LOGL, 0>(sm + (tid / TC) * SSTRIDE, tid % TC, a.tw, n >> LOGL);
    if (STEP == 0) {
        for (int idx = tid; idx < 16 * L; idx += THREADS) {
            const int cc = idx >> LOGL, k = idx & (L - 1);
            xb[(long long)(col0 + cc) * L + k] = sm[cc * SSTRIDE + pad(k)];
        }
    } else {
        const bool norm = (a.flags & SDR_FFT_NORM) != 0;
        const int out_len = (a.flags & SDR_FFT_RFFT) ? n - n / 2 : n;
        float2 *ob = a.out + b * out_len;
        for (int r = tid >> 4; r < L; r += THREADS / 16) {
            const int k = (col0 + c) + 256 * r;  // spectrum bin
            const int slot = out_slot(k, n, a.flags);
            if (slot < 0) continue;
            float2 v = sm[c * SSTRIDE + pad(r)];
            if (norm) { v.x *= a.norm; v.y *= a.norm; }
            ob[slot] = v;
        }
    }
}

// ---- n = 2^14 .. 2^16: four-step in ONE persistent launch, intermediate kept in L2 ------------------------------
// n = 256 * N2 (N2 = 64, 128, 256).  Work items of 4096 elements, handed out in ticket order:
//   STEP 0 (transform b, tile j): the 16 columns 16j.. of the [256][N2] view; 256-point FFT down each column; result
//          row-major scratch[256 c + k2] in the OUTPUT buffer.  global -> registers (radix 16) -> shared -> registers
//          (radix 16) -> global: one shared exchange, 128-byte segments on both sides.
//   STEP 1 (transform b, tile j): the NC = 4096/N2 adjacent columns k of the [N2][256] view of the scratch, element
//          (r, k) times W_n^{k r}; N2-point FFT down each column; bin k1 is X[k + 256 k1].  Reads and writes the
//          same address set, so it runs in place.
// Items are ordered wave by wave: STEP 0 of transform g, then STEP 1 of transform g - LAG, with LAG large enough that
// every resident CTA holds an earlier ticket by the time a STEP 1 item is taken.  A STEP 1 item waits (acquire spin
// on a per-transform counter that STEP 0 items bump after a release fence) for its transform's columns; tickets are
// served in order by CTAs that are all resident, so the wait always ends.  The scratch of the ~LAG transforms in
// flight (about 10 MB) never leaves the 126 MB L2: HBM sees 8 B/sample in and 8 B/sample out, as for small n.
// W_n^{k r} is generated per thread from two exact table entries (W_n^{k t}, W_n^{k TC}) by a depth-4 product tree.
template <int LOGN2> struct L2Plan {
    static constexpr int N2 = 1 << LOGN2, NC = 4096 / N2, TC = N2 / 16, R2 = N2 / 16, NB2 = 16 / R2, S = N2 / 16;
    static constexpr int SSTRIDE0 = padlen(256), SSTRIDE1 = padlen(N2);
    static constexpr int SM_ELEMS = (16 * SSTRIDE0 > NC * SSTRIDE1) ? 16 * SSTRIDE0 : NC * SSTRIDE1;
    static constexpr size_t smem_bytes() { return (size_t)(SM_ELEMS + 15 * 16 + (R2 - 1) * 16) * sizeof(float2); }
};

__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <int LOGN2, int FMT>
__global__ void __launch_bounds__(256, 4) fft_l2_kernel(FftArgs a, int lag, long long total_items) {
    using PL = L2Plan<LOGN2>;
    constexpr int N2 = PL::N2, NC = PL::NC, TC = PL::TC, R2 = PL::R2, NB2 = PL::NB2, S = PL::S;
    constexpr int n = 256 * N2;
    extern __shared__ float4 smem4[];
    __shared__ long long s_item;
    float2 *sm = reinterpret_cast<float2 *>(smem4);
    float2 *tw0 = sm + PL::SM_ELEMS;   // W_256^{q t}, q = 1..15, t < 16
    float2 *tw1 = tw0 + 15 * 16;       // W_N2^{s k}, s = 1..R2-1, k < 16
    const int tid = threadIdx.x;
    for (int i = tid; i < 15 * 16; i += 256) tw0[i] = __ldg(a.tw + (long long)((i / 16 + 1) * (i % 16)) * (n / 256));
    for (int i = tid; i < (R2 - 1) * 16; i += 256) tw1[i] = __ldg(a.tw + (long long)((i / 16 + 1) * (i % 16)) * 256);
    int *ticket = a.work, *flags = a.work + 1;
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    const int half = (a.flags & SDR_FFT_SHIFT) ? N2 / 2 : 0;
    // the next ticket is requested while the current item is processed (the atomic's round trip is off the critical path)
    long long next = 0;
    if (tid == 0) next = (long long)atomicAdd(ticket, 1);
    for (;;) {
        __syncthreads();  // s_item and the exchange buffer are free again
        if (tid == 0) {
            s_item = next;
            if (next < total_items) next = (long long)atomicAdd(ticket, 1);
        }
        __syncthreads();
        const long long item = s_item;
        if (item >= total_items) break;
        const long long g = item / (2 * S);
        const int slot = (int)(item % (2 * S));
        if (slot < S) {
            // ------------------------------ STEP 0 ------------------------------
            const long long b = g;
            if (b >= a.batches) continue;
            const int col0 = 16 * slot;
            float2 v[16];
            {
                const int c = tid & 15, rr = tid >> 4;
                const long long src = b * n + col0 + c + (long long)rr * N2;
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = load_elem<FMT>(a.in, src + (long long)e * 16 * N2);
                dft<16, 1, true>(v);
                float2 *dst = sm + c * PL::SSTRIDE0;
#pragma unroll
                for (int q = 0; q < 16; ++q) dst[17 * rr + q] = v[q];  // pad(16 rr + q) = 17 rr + q
            }
            __syncthreads();
            {
                const int col = tid >> 4, t = tid & 15;
                const float2 *srcs = sm + col * PL::SSTRIDE0;
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = srcs[t + 17 * e];  // pad(t + 16 e) = t + 17 e for t < 16
#pragma unroll
                for (int q = 1; q < 16; ++q) v[q] = cmul(v[q], tw0[(q - 1) * 16 + t]);
                dft<16, 1, true>(v);
                float2 *dst = a.out + b * n + 256LL * (col0 + col) + t;
#pragma unroll
                for (int q = 0; q < 16; ++q) dst[16 * q] = v[q];
            }
            __syncthreads();
            if (tid == 0) {
                __threadfence();  // cumulative: the whole CTA's stores (ordered before it by the barrier) are released
                atomicAdd(flags + b, 1);
            }
        } else {
            // ------------------------------ STEP 1 ------------------------------
            const long long b = g - lag;
            if (b < 0 || b >= a.batches) continue;
            if (tid == 0)
                while (ld_acquire_gpu(flags + b) < S) __nanosleep(64);
            __syncthreads();  // the acquire above + this barrier order every thread's (L2, .cg) loads after the STEP 0 stores
            const int c = tid % NC, t = tid / NC;
            const int k = NC * (slot - S) + c;
            float2 v[16];
            {
                const float2 *src = a.out + b * n + k + 256LL * t;
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = __ldcg(src + 256LL * TC * e);
                // a_e = W_n^{k (t + e TC)} = w0 * ws^e
                const float2 w0 = __ldg(a.tw + k * t), p1 = __ldg(a.tw + k * TC);
                const float2 p2 = cmul(p1, p1), p4 = cmul(p2, p2), p8 = cmul(p4, p4);
                float2 tw[16];
                tw[0] = w0; tw[1] = cmul(w0, p1); tw[2] = cmul(w0, p2); tw[3] = cmul(tw[1], p2);
#pragma unroll
                for (int e = 0; e < 4; ++e) tw[4 + e] = cmul(tw[e], p4);
#pragma unroll
                for (int e = 0; e < 8; ++e) tw[8 + e] = cmul(tw[e], p8);
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = cmul(v[e], tw[e]);
            }
            dft<16, 1, true>(v);
            float2 *col = sm + c * PL::SSTRIDE1;
#pragma unroll
            for (int q = 0; q < 16; ++q) col[17 * t + q] = v[q];  // pad(16 t + q) = 17 t + q
            __syncthreads();
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = col[pad(t + e * TC)];
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi) {
                const int kk = (t + vi * TC) & 15;
#pragma unroll
                for (int q = 1; q < R2; ++q) v[vi + q * NB2] = cmul(v[vi + q * NB2], tw1[(q - 1) * 16 + kk]);
            }
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi) dft<R2, NB2, true>(v + vi);
            float2 *ob = a.out + b * n + k;
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi)
#pragma unroll
                for (int q = 0; q < R2; ++q) {
                    const int k1 = (t + vi * TC) + 16 * q;  // bin k + 256 k1
                    float2 o = v[vi + q * NB2];
                    if (norm) { o.x *= a.norm; o.y *= a.norm; }
                    ob[256LL * ((k1 + half) & (N2 - 1))] = o;
                }
        }
    }
}

// MEASURED AND REMOVED (round 2): a software-prefetching variant of fft_l2_kernel -- tickets requested two ahead, the next
// item's 16 elements per thread loaded into registers while the current item is computed (STEP 1 items only when their
// transform's counter already reads complete) -- at 120 registers and therefore 2 CTAs per SM instead of 4.  Correct (the
// FFT suite passed) and SLOWER on every size: 180 / 177 / 170 vs 228 / 220 / 213 Gsamples/s at n = 2^14 / 2^15 / 2^16, A/B on
// one box (profiles/r02_ab_tma.txt).  ncu on the kernel below (profiles/r02_ncu_fft_l2_64k.txt): barrier stalls 6.5 and
// long-scoreboard 3.1 cycles per issue, issue 44 %, L2 44 %, DRAM 43 %: what hides the loads here is the OTHER CTAs of the
// SM, and halving their number costs more than the prefetch gains.
template <int LOGN2, int FMT>
int launch_l2(const FftArgs &a, cudaStream_t st) {
    using PL = L2Plan<LOGN2>;
    const size_t smem = PL::smem_bytes();
    auto kern = fft_l2_kernel<LOGN2, FMT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int sms = current_sm_count();
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);
    if (per_sm < 1) per_sm = 1;
    const long long resident = (long long)sms * per_sm;
    // every resident CTA holds a STEP 0 (or older) ticket before the first STEP 1 item of a transform is reached
    const int lag = (int)((resident * 3 / 2 + 2 * PL::S - 1) / (2 * PL::S)) + 1;
    const long long total = (a.batches + lag) * 2 * PL::S;
    e = cudaMemsetAsync(a.work, 0, (size_t)(a.batches + 1) * sizeof(int), st);
    if (e != cudaSuccess) return cuda_status(e);
    const long long ctas = total < resident ? total : resident;
    // FORWARD PROGRESS: a STEP 1 item spins on a counter that STEP 0 items of the same transform bump; tickets are handed
    // out in order, so the wait ends iff every CTA that holds an earlier ticket is RUNNING -- i.e. the grid must not
    // exceed what the device keeps resident at once (occupancy x SMs, queried above for this kernel and shared-memory
    // size).  Under MPS with an active-thread-percentage limit, or a partitioned GPU that reports more SMs than it gives
    // this process, that premise fails; SDR_FFT_NO_L2=1 then selects the two-launch four-step (launch_big), which has
    // no inter-CTA wait at all.
    if (ctas > resident || ctas < 1) return SDR_ERR_UNSUPPORTED;
    kern<<<(unsigned)ctas, 256, smem, st>>>(a, lag, total);
    count_launch();
    return launch_status();
}

// ---- n = 2^14 .. 2^16, round 2: the same L2-resident four-step with WARP-PRIVATE work items -----------------------
// ncu on fft_l2_kernel: barrier stalls 6.5 cycles per issue -- four CTA-wide barriers per 4096-element item, each waiting
// for the slowest warp's loads.  Here an item is 1024 elements owned by ONE warp (the fft1024_warp_kernel recipe): 32
// points per lane, a radix-32 pass in registers, one exchange through warp-private padded shared memory, a radix-LJ pass,
// so the only synchronisation is __syncwarp().  n = La * Lb (128 x 128, 256 x 128, 256 x 256):
//   STEP 0 (transform b, tile s): NCW adjacent columns of the [La][Lb] view; La-point FFT down each; result row-major
//          scratch[c La + ka] in the OUTPUT buffer.
//   STEP 1 (transform b, tile s): NCW adjacent columns ka of the [Lb][La] view of the scratch, element (c, ka) times
//          W_n^{c ka}; Lb-point FFT down each; bin kb is X[ka + La kb].  Same address set in and out: in place.
// A column of L = 32 LJ points is held by LJ lanes (LJ = 8: 4 columns per warp, LJ = 4: 8 columns per warp); lane
// (j, cl) = (lane / NCW, lane % NCW) loads rows j + LJ e (e < 32) of column cl -- every load and store instruction
// covers whole 32-byte sectors (NCW adjacent c64) -- and
//   X[k1 + 32 k2] = sum_j W_LJ^{j k2} W_L^{j k1} sum_e W_32^{e k1} x[j + LJ e].
// Items are assigned STATICALLY: in round r warp w takes item r W + ((w + rot_r) mod W) of the same wave order as above
// (STEP 0 of transform g, STEP 1 of transform g - lag); rot_r makes every warp alternate between the two (cheaper /
// dearer) steps.  A STEP 1 item acquire-spins on its transform's counter.  Forward progress: every warp walks its items
// in increasing global order and all warps are resident (grid = occupancy x SMs, checked by the launcher), so the
// lowest unfinished item always belongs to a running warp whose dependencies (lower items) are complete.
template <int LJ> struct ColPlan {
    static constexpr int NCW = 32 / LJ, NB = 32 / LJ;  // L = 32 LJ points per column
    static constexpr int SK = LJ + 1;                 // exchange: element (cl, k1, j) at cl SC + k1 SK + j
    static constexpr int SC = LJ == 8 ? 292 : 162;    // both the k1-major writes and the j-major reads conflict free
    static constexpr int XCH = NCW * SC;              // float2 per warp
};

// in: v[e] = x[j + LJ e]; out: v[i + NB k2] = X[(j + LJ i) + 32 k2]
template <int LJ, bool PK>
__device__ __forceinline__ void col_fft(float2 (&v)[32], float2 *xch, const float2 *twl, int j, int cl) {
    using CP = ColPlan<LJ>;
    float2 w[32];
    dft32<PK>(v, w);
#pragma unroll
    for (int k1 = 1; k1 < 32; ++k1) w[k1] = cmul(w[k1], twl[k1 * LJ + j]);
    float2 *wr = xch + cl * CP::SC + j;
#pragma unroll
    for (int k1 = 0; k1 < 32; ++k1) wr[k1 * CP::SK] = w[k1];
    __syncwarp();
    const float2 *rd = xch + cl * CP::SC + j * CP::SK;
#pragma unroll
    for (int i = 0; i < CP::NB; ++i)
#pragma unroll
        for (int jp = 0; jp < LJ; ++jp) v[i + CP::NB * jp] = rd[i * LJ * CP::SK + jp];
    __syncwarp();  // the exchange buffer may be rewritten by this warp's next item
#pragma unroll
    for (int i = 0; i < CP::NB; ++i) dft<LJ, CP::NB, PK>(v + i);
}

template <int LOGN> struct L2WPlan {
    static constexpr int LJA = LOGN == 14 ? 4 : 8, LJB = LOGN == 16 ? 8 : 4;
    static constexpr int LA = 32 * LJA, LB = 32 * LJB, S = (1 << LOGN) / 1024;
    static constexpr int WARPS = 8;
    static constexpr int XCH = ColPlan<LJA>::XCH > ColPlan<LJB>::XCH ? ColPlan<LJA>::XCH : ColPlan<LJB>::XCH;
    static constexpr size_t smem_bytes() { return (size_t)(WARPS * XCH + 32 * LJA + 32 * LJB) * sizeof(float2); }
};

template <int LOGN, int FMT>
__global__ void __launch_bounds__(256, 2) fft_l2w_kernel(FftArgs a, int lag, long long total_items) {
    using PL = L2WPlan<LOGN>;
    constexpr int LJA = PL::LJA, LJB = PL::LJB, LA = PL::LA, LB = PL::LB, S = PL::S, n = 1 << LOGN;
    constexpr int NCWA = 32 / LJA, NCWB = 32 / LJB;
    constexpr bool PK = true;
    extern __shared__ float4 smem4[];
    float2 *sm = reinterpret_cast<float2 *>(smem4);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    float2 *xch = sm + warp * PL::XCH;
    float2 *twa = sm + PL::WARPS * PL::XCH;  // W_La^{j k1} at [k1 LJA + j]
    float2 *twb = twa + 32 * LJA;            // W_Lb^{j k1} at [k1 LJB + j]
    for (int i = tid; i < 32 * LJA; i += 256) twa[i] = __ldg(a.tw + (long long)((i / LJA) * (i % LJA)) * (n / LA));
    for (int i = tid; i < 32 * LJB; i += 256) twb[i] = __ldg(a.tw + (long long)((i / LJB) * (i % LJB)) * (n / LB));
    __syncthreads();
    int *flags = a.work + 1;
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    const int half = (a.flags & SDR_FFT_SHIFT) ? LB / 2 : 0;
    const long long W = (long long)gridDim.x * PL::WARPS;
    const int w = blockIdx.x * PL::WARPS + warp;
    const int delta = (int)((((S - W) % (2 * S)) + 2 * S) % (2 * S));
    int rot = 0;
    for (long long base = 0; base < total_items; base += W, rot = (rot + delta) % (2 * S)) {
        long long pos = w + rot;
        if (pos >= W) pos -= W;
        const long long item = base + pos;
        if (item >= total_items) continue;
        const long long g = item / (2 * S);
        const int slot = (int)(item % (2 * S));
        float2 v[32];
        if (slot < S) {
            // ------------------------------ STEP 0 ------------------------------
            const long long b = g;
            if (b >= a.batches) continue;
            const int j = lane / NCWA, cl = lane % NCWA;
            const int c = slot * NCWA + cl;
            const long long src = b * n + (long long)j * LB + c;
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = load_elem<FMT>(a.in, src + (long long)e * LJA * LB);
            col_fft<LJA, PK>(v, xch, twa, j, cl);
            float2 *dst = a.out + b * n + (long long)c * LA + j;
#pragma unroll
            for (int i = 0; i < NCWA; ++i)
#pragma unroll
                for (int k2 = 0; k2 < LJA; ++k2) dst[LJA * i + 32 * k2] = v[i + NCWA * k2];
            __syncwarp();  // orders the other lanes' stores before lane 0's fence
            if (lane == 0) {
                __threadfence();
                atomicAdd(flags + b, 1);
            }
        } else {
            // ------------------------------ STEP 1 ------------------------------
            const long long b = g - lag;
            if (b < 0 || b >= a.batches) continue;
            const int j = lane / NCWB, cl = lane % NCWB;
            const int ka = (slot - S) * NCWB + cl;
            // twiddle W_n^{ka (j + LJB e)} = w0 p1^e, from two exact table entries by a depth-5 product tree
            float2 w0 = __ldg(a.tw + ka * j);
            const float2 p1 = __ldg(a.tw + ka * LJB);
            if (lane == 0)
                while (ld_acquire_gpu(flags + b) < S) __nanosleep(64);
            __syncwarp();  // the acquire above + this barrier order every lane's (L2, .cg) loads after the STEP 0 stores
            float2 *col = a.out + b * n + ka;
            {
                const float2 *src = col + (long long)j * LA;
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = __ldcg(src + (long long)e * LJB * LA);
            }
            // 1/sqrt(n) folds into the twiddle exactly when it is a power of two (n = 4^k)
            const bool fold = norm && (LOGN % 2 == 0);
            if (fold) { w0.x *= a.norm; w0.y *= a.norm; }
            {
                const float2 p2 = cmul(p1, p1), p4 = cmul(p2, p2), p8 = cmul(p4, p4), p16 = cmul(p8, p8);
                float2 t[32];
                t[0] = w0; t[1] = cmul(w0, p1);
#pragma unroll
                for (int e = 0; e < 2; ++e) t[2 + e] = cmul(t[e], p2);
#pragma unroll
                for (int e = 0; e < 4; ++e) t[4 + e] = cmul(t[e], p4);
#pragma unroll
                for (int e = 0; e < 8; ++e) t[8 + e] = cmul(t[e], p8);
#pragma unroll
                for (int e = 0; e < 16; ++e) t[16 + e] = cmul(t[e], p16);
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = cmul(v[e], t[e]);
            }
            col_fft<LJB, PK>(v, xch, twb, j, cl);
            const float sc = (norm && !fold) ? a.norm : 1.0f;
#pragma unroll
            for (int i = 0; i < NCWB; ++i)
#pragma unroll
                for (int k2 = 0; k2 < LJB; ++k2) {
                    const int kb = (j + LJB * i) + 32 * k2;  // bin ka + La kb
                    float2 o = v[i + NCWB * k2];
                    if (LOGN % 2 != 0) { o.x *= sc; o.y *= sc; }
                    col[(long long)LA * ((kb + half) & (LB - 1))] = o;
                }
        }
    }
}

template <int LOGN, int FMT>
int launch_l2w(const FftArgs &a, cudaStream_t st) {
    using PL = L2WPlan<LOGN>;
    const size_t smem = PL::smem_bytes();
    auto kern = fft_l2w_kernel<LOGN, FMT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int sms = current_sm_count();
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);
    if (per_sm < 1) return SDR_ERR_UNSUPPORTED;
    const long long resident = (long long)sms * per_sm;  // every CTA of the grid must be running: see FORWARD PROGRESS above
    const long long W = resident * PL::WARPS;
    // a STEP 1 item comes at least one and a half rounds after the STEP 0 items of its transform
    const int lag = (int)((W * 3 / 2 + 2 * PL::S - 1) / (2 * PL::S)) + 1;
    const long long total = (a.batches + lag) * 2 * PL::S;
    e = cudaMemsetAsync(a.work, 0, (size_t)(a.batches + 1) * sizeof(int), st);
    if (e != cudaSuccess) return cuda_status(e);
    kern<<<(unsigned)resident, 256, smem, st>>>(a, lag, total);
    count_launch();
    return launch_status();
}

// ---- n = 2^14 .. 2^16, round 2: fft_l2_kernel fed by TMA ----------------------------------------------------------
// ncu on fft_l2_kernel: barrier 6.5 + long scoreboard 3.1 stall cycles per issue -- every item starts with 16 exposed
// LDG.64 per thread and the CTA's first barrier waits for the slowest warp's loads.  (A warp-private variant with 32
// points per lane, fft_l2w_kernel above, removes the barriers but needs rows of 4 adjacent c64 = one 32-byte sector per
// row and warp: 8 L1 wavefronts per request instead of 2, L1TEX 69 % busy, 165 vs 225 Gsamples/s: kept for the record.)
// Here the NEXT item's 4096-element tile is copied into a second shared-memory stage by ONE TMA tensor copy
// (cp.async.bulk.tensor.3d over {columns, rows, transforms}, SASS UTMALDG, issued by one thread, completing in bytes on
// an mbarrier; first version: 256 bulk row copies of 128 bytes per item -- 27 cycles each in the copy engine, 85
// Gsamples/s) while the current item is computed:
// an item's first pass reads shared memory instead of HBM / L2, the same number of issued instructions (LDS for LDG).
// The consumed stage doubles as the item's exchange buffer.  Items are assigned statically (round it: item
// it G + ((x + rot_it) mod G), rot_it alternating the two steps on every CTA), so the next item is known without a
// ticket, and a CTA-wide barrier serves three purposes at once (stage consumed / previous item's stores done -> its
// counter bump / other stage free for the next copy): two barriers per item instead of four.
// Forward progress: as for fft_l2w_kernel -- a CTA walks its items in increasing global order, a STEP 1 copy waits only
// for STEP 0 items at least lag 2S - S items older, and lag 2S > G + 3S makes those older than anything this CTA has
// not yet signalled; the launcher keeps the whole grid resident.
template <int LOGN2, int FMT>
__global__ void __launch_bounds__(288, 3) fft_l2t_kernel(FftArgs a, int lag, long long total_items,
                                                         const __grid_constant__ CUtensorMap map_in,
                                                         const __grid_constant__ CUtensorMap map_scr) {
    using PL = L2Plan<LOGN2>;
    constexpr int N2 = PL::N2, NC = PL::NC, TC = PL::TC, R2 = PL::R2, NB2 = PL::NB2, S = PL::S;
    constexpr int n = 256 * N2, ES = FmtBytes<FMT>::v;
    constexpr int STAGE = (PL::SM_ELEMS + 15) & ~15;  // float2 per stage (128-byte multiple)
    extern __shared__ __align__(128) float4 smem_l2t[];  // TMA tensor copies land on 128-byte boundaries
    __shared__ __align__(8) uint64_t full_bar[2];
    __shared__ unsigned cnt[2];
    float2 *sm = reinterpret_cast<float2 *>(smem_l2t);
    float2 *tw0 = sm + 2 * STAGE;      // W_256^{q t}, q = 1..15, t < 16
    float2 *tw1 = tw0 + 15 * 16;       // W_N2^{s k}, s = 1..R2-1, k < 16
    const int tid = threadIdx.x;
    for (int i = tid; i < 15 * 16; i += 288) tw0[i] = __ldg(a.tw + (long long)((i / 16 + 1) * (i % 16)) * (n / 256));
    for (int i = tid; i < (R2 - 1) * 16; i += 288) tw1[i] = __ldg(a.tw + (long long)((i / 16 + 1) * (i % 16)) * 256);
    if (tid == 0) {
        mbar_init(smem_u32(&full_bar[0]), 1);
        mbar_init(smem_u32(&full_bar[1]), 1);
        mbar_init_fence();
        cnt[0] = 0;
        cnt[1] = 0;
    }
    __syncthreads();
    int *flags = a.work + 1;
    const bool norm = (a.flags & SDR_FFT_NORM) != 0;
    const int half = (a.flags & SDR_FFT_SHIFT) ? N2 / 2 : 0;
    const long long G = gridDim.x;
    const int x = blockIdx.x;
    const int delta = (int)((((S - G) % (2 * S)) + 2 * S) % (2 * S));
    const long long n_it = (total_items + G - 1) / G;
    auto item_at = [&](long long it) -> long long {
        long long pos = x + (int)((it * delta) % (2 * S));
        if (pos >= G) pos -= G;
        return it * G + pos;
    };
    // item -> (step, transform, tile); b < 0: nothing to do
    auto decode = [&](long long item, bool &step1, long long &b, int &tile) {
        const long long g = item / (2 * S);
        const int slot = (int)(item % (2 * S));
        step1 = slot >= S;
        tile = step1 ? slot - S : slot;
        b = step1 ? g - lag : g;
        if (item >= total_items || b >= a.batches) b = -1;
    };
    // service lane: copy an item's tile into stage s.  STEP 0 tile: 256 rows x 16 elements of the input; STEP 1 tile:
    // N2 rows x NC c64 of the scratch, after its transform's STEP 0 items have all signalled (try_only: give up instead
    // of spinning; returns false when the copy was not issued)
    auto load_item = [&](long long item, int s, bool try_only) -> bool {
        bool step1; long long b; int tile;
        decode(item, step1, b, tile);
        if (b < 0) return true;
        const uint32_t bar = smem_u32(&full_bar[s]), dst = smem_u32(sm + (size_t)s * STAGE);
        if (!step1) {
            mbar_arrive_expect_tx(bar, 4096 * ES);
            tma_load_3d(dst, &map_in, 16 * tile, 0, (int)b, bar);
        } else {
            while (ld_acquire_gpu(flags + b) < S) {
                if (try_only) return false;
                __nanosleep(64);
            }
            // the STEP 0 stores (generic proxy, other SMs; acquired above) before this thread's async-proxy reads of them
            fence_proxy_async_all();
            mbar_arrive_expect_tx(bar, 4096 * 8);
            tma_load_3d(dst, &map_scr, NC * tile, 0, (int)b, bar);
        }
        return true;
    };
    // monotonic shared counters, one release-add per compute warp and item: cnt[0] = "exchange read, the stage is free",
    // cnt[1] = "stores issued".  (Counters, not barrier phases: the compute warps may run up to two items ahead of the
    // service lane, which a parity cannot express.)
    auto cnt_arrive = [&](int which) {
        __syncwarp();  // orders the other lanes' accesses before lane 0's release
        if ((tid & 31) == 0)
            asm volatile("red.release.cta.shared::cta.add.u32 [%0], 1;" ::"r"(smem_u32(&cnt[which])) : "memory");
    };
    auto cnt_wait = [&](int which, unsigned target) {
        unsigned v;
        for (;;) {
            asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(&cnt[which])) : "memory");
            if (v >= target) break;
            __nanosleep(32);
        }
    };

    // ---- service warp (one lane): everything that waits on the memory system without computing -- the TMA issue, the
    // acquire spin on a STEP 1 item's counter, the release fence + counter bump behind an item's stores.  With thread 0
    // of the compute warps doing this (first version: 5.5 barrier-stall cycles per issue) seven warps sat at barrier (B)
    // for the whole of warp 0's fence.  Item it + 2's tile is requested as soon as item it's exchange has been read
    // (its stage is free): a copy has one and a half items to land.
    if (tid >= 256) {
        if (tid != 256) return;
        load_item(item_at(0), 0, false);
        if (n_it > 1) load_item(item_at(1), 1, false);
        unsigned nvalid = 0;
        for (long long it = 0; it < n_it; ++it) {
            bool step1; long long b; int tile;
            decode(item_at(it), step1, b, tile);
            if (b >= 0) {
                ++nvalid;
                cnt_wait(0, 8 * nvalid);
            }
            bool issued = true;
            if (it + 2 < n_it) issued = load_item(item_at(it + 2), (int)(it & 1), true);
            if (b >= 0 && !step1) {
                cnt_wait(1, 8 * nvalid);
                __threadfence();  // cumulative: the CTA's stores of this item (acquired from the warps' release-adds)
                atomicAdd(flags + b, 1);
            }
            if (!issued) load_item(item_at(it + 2), (int)(it & 1), false);
        }
        return;
    }
    uint32_t ph = 0;        // bit s = parity of stage s's next completion
    for (long long it = 0; it < n_it; ++it) {
        const int s = (int)(it & 1);
        float2 *st = sm + (size_t)s * STAGE;
        bool step1; long long b; int tile;
        decode(item_at(it), step1, b, tile);
        float2 v[16];
        if (b >= 0) {
            if (!step1) {
                mbar_wait(smem_u32(&full_bar[s]), (ph >> s) & 1u);
                const int c = tid & 15, rr = tid >> 4;
                const unsigned char *raw = reinterpret_cast<const unsigned char *>(st);
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = raw_elem<FMT>(raw, (rr + 16 * e) * 16 + c);
            } else {
                const int c = tid % NC, t = tid / NC;
                const int k = NC * tile + c;
                // a_e = W_n^{k (t + e TC)} = w0 * ws^e (the two table loads are in flight while the tile lands)
                const float2 w0 = __ldg(a.tw + k * t), p1 = __ldg(a.tw + k * TC);
                mbar_wait(smem_u32(&full_bar[s]), (ph >> s) & 1u);
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = st[(t + TC * e) * NC + c];
                const float2 p2 = cmul(p1, p1), p4 = cmul(p2, p2), p8 = cmul(p4, p4);
                float2 tw[16];
                tw[0] = w0; tw[1] = cmul(w0, p1); tw[2] = cmul(w0, p2); tw[3] = cmul(tw[1], p2);
#pragma unroll
                for (int e = 0; e < 4; ++e) tw[4 + e] = cmul(tw[e], p4);
#pragma unroll
                for (int e = 0; e < 8; ++e) tw[8 + e] = cmul(tw[e], p8);
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = cmul(v[e], tw[e]);
            }
            ph ^= 1u << s;
            dft<16, 1, true>(v);
        }
        if (b < 0) continue;
        asm volatile("bar.sync 1, 256;" ::: "memory");  // (A) the tile is in registers: the stage becomes the exchange buffer
        if (!step1) {
            {
                const int c = tid & 15, rr = tid >> 4;
                float2 *dst = st + c * PL::SSTRIDE0;
#pragma unroll
                for (int q = 0; q < 16; ++q) dst[17 * rr + q] = v[q];  // pad(16 rr + q) = 17 rr + q
            }
            asm volatile("bar.sync 2, 256;" ::: "memory");  // (B) compute warps only
            const int col = tid >> 4, t = tid & 15;
            const float2 *srcs = st + col * PL::SSTRIDE0;
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = srcs[t + 17 * e];  // pad(t + 16 e) = t + 17 e for t < 16
            fence_proxy_async();  // these accesses before the stage's next tensor copy
            cnt_arrive(0);
#pragma unroll
            for (int q = 1; q < 16; ++q) v[q] = cmul(v[q], tw0[(q - 1) * 16 + t]);
            dft<16, 1, true>(v);
            float2 *dst = a.out + b * n + 256LL * (16 * tile + col) + t;
#pragma unroll
            for (int q = 0; q < 16; ++q) dst[16 * q] = v[q];
            cnt_arrive(1);
        } else {
            const int c = tid % NC, t = tid / NC;
            const int k = NC * tile + c;
            float2 *col = st + c * PL::SSTRIDE1;
#pragma unroll
            for (int q = 0; q < 16; ++q) col[17 * t + q] = v[q];  // pad(16 t + q) = 17 t + q
            asm volatile("bar.sync 2, 256;" ::: "memory");  // (B)
#pragma unroll
            for (int e = 0; e < 16; ++e) v[e] = col[pad(t + e * TC)];
            fence_proxy_async();
            cnt_arrive(0);
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi) {
                const int kk = (t + vi * TC) & 15;
#pragma unroll
                for (int q = 1; q < R2; ++q) v[vi + q * NB2] = cmul(v[vi + q * NB2], tw1[(q - 1) * 16 + kk]);
            }
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi) dft<R2, NB2, true>(v + vi);
            float2 *ob = a.out + b * n + k;
#pragma unroll
            for (int vi = 0; vi < NB2; ++vi)
#pragma unroll
                for (int q = 0; q < R2; ++q) {
                    const int k1 = (t + vi * TC) + 16 * q;  // bin k + 256 k1
                    float2 o = v[vi + q * NB2];
                    if (norm) { o.x *= a.norm; o.y *= a.norm; }
                    ob[256LL * ((k1 + half) & (N2 - 1))] = o;
                }
            cnt_arrive(1);
        }
    }
}

// {cols, rows, transforms} view of `batches` transforms of rows x cols elements of `es` bytes; box = cols_box x rows x 1
inline bool fft_tile_map(CUtensorMap *tm, const void *base, int es, int cols, int rows, long long batches, int cols_box) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const CUtensorMapDataType dt = es == 8 ? CU_TENSOR_MAP_DATA_TYPE_UINT64 : es == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16;
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batches};
    cuuint64_t strides[2] = {(cuuint64_t)cols * es, (cuuint64_t)cols * rows * es};  // bytes, dims 1..2
    cuuint32_t box[3] = {(cuuint32_t)cols_box, (cuuint32_t)rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    return enc(tm, dt, 3, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int LOGN2, int FMT>
int launch_l2t(const FftArgs &a, cudaStream_t st) {
    using PL = L2Plan<LOGN2>;
    const size_t smem = (size_t)(2 * ((PL::SM_ELEMS + 15) & ~15) + 15 * 16 + (PL::R2 - 1) * 16) * sizeof(float2);
    auto kern = fft_l2t_kernel<LOGN2, FMT>;
    CUtensorMap map_in, map_scr;
    if (!fft_tile_map(&map_in, a.in, FmtBytes<FMT>::v, PL::N2, 256, a.batches, 16) ||
        !fft_tile_map(&map_scr, a.out, 8, 256, PL::N2, a.batches, PL::NC))
        return launch_l2<LOGN2, FMT>(a, st);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_status(e);
    const int sms = current_sm_count();
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 288, smem);
    if (per_sm < 1) return SDR_ERR_UNSUPPORTED;
    const long long G = (long long)sms * per_sm;  // the whole grid resident: see FORWARD PROGRESS
    // a STEP 1 tile is requested one and a half items ahead: three rounds behind its transform's STEP 0 items
    // (SDR_FFT_L2_LAG = tenths of a round: tuning knob)
    static const int lag10 = std::getenv("SDR_FFT_L2_LAG") ? std::atoi(std::getenv("SDR_FFT_L2_LAG")) : 30;
    const int lag = (int)((G * lag10 / 10 + 2 * PL::S - 1) / (2 * PL::S)) + 1;
    const long long total = (a.batches + lag) * 2 * PL::S;
    e = cudaMemsetAsync(a.work, 0, (size_t)(a.batches + 1) * sizeof(int), st);
    if (e != cudaSuccess) return cuda_status(e);
    kern<<<(unsigned)G, 288, smem, st>>>(a, lag, total, map_in, map_scr);  // 8 compute warps + the service warp
    count_launch();
    return launch_status();
}

// ---- tiny sizes: direct DFT, one thread per output bin ---------------------------------------
template <int FMT>
__global__ void fft_naive_kernel(const void *in, float2 *out, const float2 *__restrict__ tw, long long batches,
                                 int n, unsigned flags, float norm) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    if (gid >= batches * out_len) return;
    const long long b = gid / out_len;
    const int j = (int)(gid % out_len);
    int k = j;
    if (!(flags & SDR_FFT_RFFT) && (flags & SDR_FFT_SHIFT)) {
        k = j - n / 2;
        if (k < 0) k += n;
    }
    float2 acc = make_float2(0.0f, 0.0f);
    int ph = 0;
    for (int i = 0; i < n; ++i) {
        const float2 x = load_elem<FMT>(in, b * n + i);
        acc = cadd(acc, cmul(x, __ldg(tw + ph)));
        ph += k;
        if (ph >= n) ph -= n;
    }
    if (flags & SDR_FFT_NORM) { acc.x *= norm; acc.y *= norm; }
    out[gid] = acc;
}

template <int LOGN, int FMT>
int launch_cta(const FftArgs &a, cudaStream_t st) {
    constexpr int N = 1 << LOGN, TC = N / 16;
    constexpr int THREADS = TC > 256 ? TC : 256;
    constexpr int SEQ = THREADS / TC;
    const size_t smem = (size_t)SEQ * padlen(N) * sizeof(float2);
    auto kern = fft_cta_kernel<LOGN, FMT>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
    }
    const long long ctas = (a.batches + SEQ - 1) / SEQ;
    kern<<<(unsigned)ctas, THREADS, smem, st>>>(a);
    count_launch();
    return launch_status();
}

template <int FMT>
int launch_big(const FftArgs &a, cudaStream_t st) {
    const int n = 1 << a.log_n, M = n >> 8;
    if ((a.flags & SDR_FFT_RFFT) != 0) return SDR_ERR_UNSUPPORTED;  // in-place scratch needs n outputs per row
    {
        const size_t smem = (size_t)16 * padlen(256) * sizeof(float2);
        const long long ctas = a.batches * (M / 16);
        fft_cols_kernel<8, FMT, 0><<<(unsigned)ctas, 256, smem, st>>>(a);
        count_launch();
        int rc = launch_status();
        if (rc) return rc;
    }
    const long long ctas = a.batches * 16;
    if (M == 128) {
        const size_t smem = (size_t)16 * padlen(128) * sizeof(float2);
        fft_cols_kernel<7, FMT, 1><<<(unsigned)ctas, 128, smem, st>>>(a);
    } else {
        const size_t smem = (size_t)16 * padlen(256) * sizeof(float2);
        fft_cols_kernel<8, FMT, 1><<<(unsigned)ctas, 256, smem, st>>>(a);
    }
    count_launch();
    return launch_status();
}

// smallest log2 n that takes the L2-resident four-step kernel (tuning knob: SDR_FFT_L2_MIN=13 tries it for n = 8192)
inline int l2_min_logn() {
    static int v = 0;
    if (!v) {
        const char *e = std::getenv("SDR_FFT_L2_MIN");
        v = e ? std::atoi(e) : 14;
        if (v < 13) v = 13;
    }
    return v;
}

inline bool no_l2() {
    static const bool v = std::getenv("SDR_FFT_NO_L2") != nullptr;
    return v;
}
// A/B switch SDR_FFT_L2_MODE: 0 = round 1's ticket kernel (fft_l2_kernel), 1 = warp items (fft_l2w_kernel),
// 2 = TMA-fed CTA items (fft_l2t_kernel, default)
inline int l2_mode() {
    static const int v = std::getenv("SDR_FFT_L2_MODE") ? std::atoi(std::getenv("SDR_FFT_L2_MODE")) : 2;
    return v;
}
template <int LOGN, int FMT>
int launch_l2_any(const FftArgs &a, cudaStream_t st) {
    const int mode = l2_mode();
    if (mode == 1) return launch_l2w<LOGN, FMT>(a, st);
    if (mode == 2 && (((uintptr_t)a.in) & 15) == 0) return launch_l2t<LOGN - 8, FMT>(a, st);  // bulk copies need 16-byte rows
    return launch_l2<LOGN - 8, FMT>(a, st);
}

template <int FMT>
int launch_fmt(const FftArgs &a, cudaStream_t st) {
    switch (a.log_n) {
        case 4: return launch_cta<4, FMT>(a, st);
        case 5: return launch_cta<5, FMT>(a, st);
        case 6: return launch_cta<6, FMT>(a, st);
        case 7: return launch_cta<7, FMT>(a, st);
        case 8: return launch_reg2<8, FMT>(a, st);
        case 9: return launch_reg2<9, FMT>(a, st);
        case 10:
            // 1/sqrt(1024) = 2^-5 folds exactly; the warp kernel handles U8IQ and C64 without RFFT
            if (FMT != SDR_FMT_F32 && !(a.flags & SDR_FFT_RFFT) && (((uintptr_t)a.in) & 15) == 0)
                return launch_w1k<FMT>(a, st);
            return launch_cta<10, FMT>(a, st);
        case 11: return launch_reg2<11, FMT>(a, st);
        case 12: return launch_reg2<12, FMT>(a, st);
        case 13:
            if (a.work && !(a.flags & SDR_FFT_RFFT) && l2_min_logn() <= 13) return launch_l2<5, FMT>(a, st);
            return launch_reg2<13, FMT>(a, st);
        case 14:
            if (a.work && !(a.flags & SDR_FFT_RFFT) && !no_l2())
                return launch_l2_any<14, FMT>(a, st);
            return launch_cta<14, FMT>(a, st);
        case 15:
            if (a.work && !(a.flags & SDR_FFT_RFFT) && !no_l2())
                return launch_l2_any<15, FMT>(a, st);
            return launch_big<FMT>(a, st);
        case 16:
            if (a.work && !(a.flags & SDR_FFT_RFFT) && !no_l2())
                return launch_l2_any<16, FMT>(a, st);
            return launch_big<FMT>(a, st);
    }
    return SDR_ERR_UNSUPPORTED;
}

}  // namespace

int fft_pow2_launch(const FftArgs &a, cudaStream_t st) {
    if (a.batches <= 0) return SDR_OK;
    if (a.batches > 0x7fffffffLL) return SDR_ERR_INVALID_ARG;
    switch (a.fmt) {
        case SDR_FMT_U8IQ: return launch_fmt<SDR_FMT_U8IQ>(a, st);
        case SDR_FMT_C64: return launch_fmt<SDR_FMT_C64>(a, st);
        case SDR_FMT_F32: return launch_fmt<SDR_FMT_F32>(a, st);
    }
    return SDR_ERR_INVALID_ARG;
}

int fft_naive_launch(const void *in, float2 *out, const float2 *tw, long long batches, int n, int fmt,
                     unsigned flags, float norm, cudaStream_t st) {
    if (batches <= 0 || n <= 0) return SDR_OK;
    const int out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    const long long total = batches * out_len;
    const unsigned grid = (unsigned)((total + 127) / 128);
    if (fmt == SDR_FMT_U8IQ)
        fft_naive_kernel<SDR_FMT_U8IQ><<<grid, 128, 0, st>>>(in, out, tw, batches, n, flags, norm);
    else if (fmt == SDR_FMT_C64)
        fft_naive_kernel<SDR_FMT_C64><<<grid, 128, 0, st>>>(in, out, tw, batches, n, flags, norm);
    else
        fft_naive_kernel<SDR_FMT_F32><<<grid, 128, 0, st>>>(in, out, tw, batches, n, flags, norm);
    count_launch();
    return launch_status();
}

// ---- lengths beyond the single-launch kernels (n = 2^17 .. 2^27): N = N1 * N2, the textbook four-step through global
// memory.  fft::fft transforms a WHOLE finite signal in one call (src/fft.rs:8: e.g. take(0.1) at 1.8 MS/s = 180 000
// samples -> Bluestein with m = 2^19), so this path has to exist; it is one transform per call and not a throughput
// target.  out[c][r] = in[r][c] * W_N^{r c} (tw_n != 0) -- a tiled transpose with the twiddle evaluated in f64
// (sincospi of the exactly reduced r*c mod N) and rounded once, as the table twiddles of the other kernels are.
__global__ void fft_transpose_kernel(const float2 *__restrict__ in, float2 *__restrict__ out, int rows, int cols,
                                     long long tw_n) {
    __shared__ float2 tile[32][33];
    const long long boff = (long long)blockIdx.z * rows * cols;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        if (r < rows && c < cols) tile[j][threadIdx.x] = in[boff + (long long)r * cols + c];
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) {
            float2 v = tile[threadIdx.x][j];
            if (tw_n) {
                const long long q = ((long long)r * c) % tw_n;
                double sn, cs;
                sincospi(-2.0 * (double)q / (double)tw_n, &sn, &cs);
                v = cmul(v, make_float2((float)cs, (float)sn));
            }
            out[boff + (long long)c * rows + r] = v;
        }
    }
}

static int transpose_launch(const float2 *in, float2 *out, int rows, int cols, long long tw_n, long long batches,
                            cudaStream_t st) {
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32), (unsigned)batches);
    fft_transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(in, out, rows, cols, tw_n);
    count_launch();
    return launch_status();
}

int fft_huge_launch(const float2 *in, float2 *out, float2 *s1, float2 *s2, const float2 *tw1, const float2 *tw2,
                    int log_n, long long batches, int *work, cudaStream_t st) {
    if (log_n < 17 || log_n > 27 || batches <= 0 || batches > 65535) return SDR_ERR_UNSUPPORTED;
    const int l1 = log_n / 2, l2 = log_n - l1;  // both in [8, 14]
    const int N1 = 1 << l1, N2 = 1 << l2;
    const long long N = 1LL << log_n;
    // x viewed as [N1][N2] (n = n1 N2 + n2).  (1) s1[n2][n1] = x[n1][n2]
    int rc = transpose_launch(in, s1, N1, N2, 0, batches, st);
    if (rc) return rc;
    // (2) N2 * batches transforms of length N1 over n1: s2[n2][k1]
    FftArgs a;
    a.in = s1; a.out = s2; a.tw = tw1; a.batches = batches * N2; a.log_n = l1; a.fmt = SDR_FMT_C64; a.flags = 0;
    a.norm = 1.0f; a.work = (l1 >= 14) ? work : nullptr;
    rc = fft_pow2_launch(a, st);
    if (rc) return rc;
    // (3) s1[k1][n2] = s2[n2][k1] * W_N^{n2 k1}
    rc = transpose_launch(s2, s1, N2, N1, N, batches, st);
    if (rc) return rc;
    // (4) N1 * batches transforms of length N2 over n2: s2[k1][k2]
    a.in = s1; a.out = s2; a.tw = tw2; a.batches = batches * N1; a.log_n = l2; a.work = (l2 >= 14) ? work : nullptr;
    rc = fft_pow2_launch(a, st);
    if (rc) return rc;
    // (5) X[k1 + N1 k2] = s2[k1][k2]
    return transpose_launch(s2, out, N1, N2, 0, batches, st);
}

// format conversion in front of / post-processing behind the multi-launch paths (same element rules as the fused kernels)
template <int FMT>
__global__ void fft_convert_kernel(const void *in, float2 *a, long long total) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid < total) a[gid] = load_elem<FMT>(in, gid);
}
__global__ void fft_finish_kernel(const float2 *a, float2 *out, long long batches, long long n, unsigned flags, float norm) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    if (gid >= batches * out_len) return;
    const long long b = gid / out_len, j = gid % out_len;
    long long k = j;
    // fft.rs:18-25: out[i] = X[(i - n/2) mod n]; rfft drops the first n/2 of those, leaving bins 0 .. n - n/2 - 1
    if (!(flags & SDR_FFT_RFFT) && (flags & SDR_FFT_SHIFT)) { k = j - n / 2; if (k < 0) k += n; }
    float2 v = a[b * n + k];
    if (flags & SDR_FFT_NORM) { v.x *= norm; v.y *= norm; }
    out[gid] = v;
}
int fft_convert_launch(const void *in, float2 *a, long long total, int fmt, cudaStream_t st) {
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (fmt == SDR_FMT_U8IQ) fft_convert_kernel<SDR_FMT_U8IQ><<<grid, 256, 0, st>>>(in, a, total);
    else if (fmt == SDR_FMT_C64) fft_convert_kernel<SDR_FMT_C64><<<grid, 256, 0, st>>>(in, a, total);
    else fft_convert_kernel<SDR_FMT_F32><<<grid, 256, 0, st>>>(in, a, total);
    count_launch();
    return launch_status();
}
int fft_finish_launch(const float2 *a, float2 *out, long long batches, long long n, unsigned flags, float norm,
                      cudaStream_t st) {
    const long long out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    fft_finish_kernel<<<(unsigned)((batches * out_len + 255) / 256), 256, 0, st>>>(a, out, batches, n, flags, norm);
    count_launch();
    return launch_status();
}

// ---- Bluestein (chirp-z) stages for arbitrary n: X[k] = conj(w[k]) * sum_j (x[j] conj(w[j])) w[k-j],
// w[j] = e^{+i pi j^2 / n}.  chirp[j] holds conj(w[j]) = e^{-i pi j^2/n}.
template <int FMT>
__global__ void bluestein_pre_kernel(const void *in, float2 *a, const float2 *__restrict__ chirp,
                                     long long batches, int n, int m) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= batches * m) return;
    const long long b = gid / m;
    const int j = (int)(gid % m);
    float2 v = make_float2(0.0f, 0.0f);
    if (j < n) v = cmul(load_elem<FMT>(in, b * n + j), __ldg(chirp + j));
    a[gid] = v;
}
__global__ void bluestein_mul_kernel(float2 *a, const float2 *__restrict__ bfft, long long batches, int m) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= batches * m) return;
    const int j = (int)(gid % m);
    // conj() here and in the post stage turn the second forward FFT into an inverse one
    const float2 p = cmul(a[gid], __ldg(bfft + j));
    a[gid] = make_float2(p.x, -p.y);
}
__global__ void bluestein_post_kernel(const float2 *a, float2 *out, const float2 *__restrict__ chirp,
                                      long long batches, int n, int m, unsigned flags, float norm) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    if (gid >= batches * out_len) return;
    const long long b = gid / out_len;
    const int j = (int)(gid % out_len);
    int k = j;
    if (!(flags & SDR_FFT_RFFT) && (flags & SDR_FFT_SHIFT)) {
        k = j - n / 2;
        if (k < 0) k += n;
    }
    const float2 y = a[b * m + k];
    const float inv_m = 1.0f / (float)m;
    float2 v = cmul(make_float2(y.x * inv_m, -y.y * inv_m), __ldg(chirp + k));
    if (flags & SDR_FFT_NORM) { v.x *= norm; v.y *= norm; }
    out[gid] = v;
}

int bluestein_pre_launch(const void *in, float2 *a, const float2 *chirp, long long batches, int n, int m, int fmt,
                         cudaStream_t st) {
    const long long total = batches * m;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (fmt == SDR_FMT_U8IQ) bluestein_pre_kernel<SDR_FMT_U8IQ><<<grid, 256, 0, st>>>(in, a, chirp, batches, n, m);
    else if (fmt == SDR_FMT_C64) bluestein_pre_kernel<SDR_FMT_C64><<<grid, 256, 0, st>>>(in, a, chirp, batches, n, m);
    else bluestein_pre_kernel<SDR_FMT_F32><<<grid, 256, 0, st>>>(in, a, chirp, batches, n, m);
    count_launch();
    return launch_status();
}
int bluestein_mul_launch(float2 *a, const float2 *bfft, long long batches, int m, cudaStream_t st) {
    const long long total = batches * m;
    bluestein_mul_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(a, bfft, batches, m);
    count_launch();
    return launch_status();
}
int bluestein_post_launch(const float2 *a, float2 *out, const float2 *chirp, long long batches, int n, int m,
                          unsigned flags, float norm, cudaStream_t st) {
    const int out_len = (flags & SDR_FFT_RFFT) ? n - n / 2 : n;
    const long long total = batches * out_len;
    bluestein_post_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(a, out, chirp, batches, n, m, flags, norm);
    count_launch();
    return launch_status();
}

}  // namespace sdr

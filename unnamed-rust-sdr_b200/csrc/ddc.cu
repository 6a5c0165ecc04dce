// ddc.cu -- K7, sdr_ddc_*: digital down-converter bank.  C channels of one IQ stream, each mixed to 0 Hz by its own
// 64-bit NCO, low-pass filtered and decimated by the shared D, in one pass over the input.
//
// Channel k (taps h_k, NCO increment Delta_k), input x[n] with n counted from the handle's first sample, x[<0] = 0:
//     z_k[n] = x[n] e^{-2 pi i phi_k(F + n) / 2^64},  phi_k(N) = N Delta_k mod 2^64,  F = first_sample
//     y_k[m] = sum_{j<L} h_k[j] z_k[N_m - j],  N_m = (m + 1) D - 1          (Fir::apply + Decimate, fir.rs:23-32,
//                                                                           adapters/mod.rs:30-37)
// computed as the equivalent frequency-translating FIR
//     y_k[m] = e^{-2 pi i phi_k(F + N_m) / 2^64} sum_j g_k[j] x[N_m - j],  g_k[j] = h_k[j] e^{+2 pi i (j Delta_k mod 2^64) / 2^64}
// (exact because (N - j) Delta = N Delta - j Delta mod 2^64).
//
// Two kernels:
//   ddc_tc_kernel       u8 IQ, D | 32, L <= 511: K5's integer Toeplitz GEMM (fir_umma.cu) with the channels of a group
//                       side by side along N.  Rows are 32 samples apart and every candidate of a row is kept (PC = 32 / D
//                       per channel), so the B block of a group is the channels' fir_umma_build_tables blocks (complex
//                       taps g_k) concatenated in 8-column core-matrix units.  The epilogue combines the digits as K5
//                       does, derotates and stores channel-major rows.
//   ddc_general_kernel  everything else (c64 input, L > 511, D not dividing 32, SDR_DDC_GENERAL_KERNEL): one thread per
//                       output and per 8 channels, complex FMA chain in ascending j, derotation from the exact phase.
//
// Derotation without a sincos per output.  Tiles are 4096 samples (128 rows) anchored on ABSOLUTE stream indices:
// tile boundaries sit at N - eps = 0 mod 4096 with eps = F mod D, so every kept output of a tile has N - N_tile in
// {D j + D - 1}, and
//     e^{-2 pi i phi(N)} = base(N_tile) * tab[j],   tab[j] = e^{-2 pi i ((D j + D - 1) Delta mod 2^64) / 2^64},  j < 4096 / D
// base is one f64 sincospi per tile and channel (computed by the lanes of each epilogue warp in parallel), tab is a
// per-channel f32 table built on the host in f64: two complex multiplies per output.  Everything depends on N alone,
// so the results are bit-identical across blockings, pointer alignments and halo shards with the same F mod D.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "kernels.h"
#include "nco.cuh"
#include "ptx.cuh"

using namespace sdr;

namespace {

constexpr size_t DDC_MAX_CH = 256;
constexpr int DDC_MAX_TC_K = 511;                    // K5's exactness bound for the s32 digit sums
constexpr int DDC_TILE = 4096;                       // samples per tile = 128 rows of 32
constexpr int DDC_STAGES = 4;                        // at most; fewer when the group's table leaves less shared memory
constexpr int DDC_PROD_WARPS = 3;
constexpr int DDC_MMA_WARP = DDC_PROD_WARPS;
constexpr int DDC_EPI_WARP0 = DDC_PROD_WARPS + 1;   // 16 epilogue warps: 2 accumulator sets x 2 channel halves x 4 quadrants
constexpr int DDC_THREADS = (DDC_PROD_WARPS + 1 + 16) * 32;
constexpr int DDC_ACC_COLS = 256;                    // TMEM columns per accumulator set (two sets fill the 512)
constexpr size_t DDC_SMEM_MAX = 220 * 1024;
constexpr size_t DDC_SLAB_BYTES = (size_t)32 << 20;  // host-memory calls: input chunk size

// stage = the window starts of one tile's 128 rows (64 bytes apart) + the KS * 32-byte halo of the last row
__host__ __device__ constexpr int ddc_stage_bytes(int KS) { return (64 * 127 + 32 * KS + 1023) / 1024 * 1024; }
__host__ __device__ constexpr size_t ddc_smem_bytes(int KS, int Ng, int stages) {
    return (size_t)KS * Ng * 32 + (size_t)stages * ddc_stage_bytes(KS) + 1024 + 256;
}

struct DdcChan {        // per channel: K5's epilogue constants of its table
    int c10[2], m2[2];  // -(256 C1 + C0) and 0x4B400000 - C2, per part
    float sc0, sc2;     // 2^-(S+7) * {1, 65536}
};

struct DdcTcArgs {
    const uint8_t *in, *hist;  // caller block (n_in samples), carried history (HL samples, newest last)
    long long n_in, hist_valid;  // hist_valid = history samples that belong to the stream
    int HL;
    const uint8_t *tab;        // this call's alignment variant: ngroups blocks of KS * Ng * 32 bytes
    const DdcChan *chan;
    const float2 *rot;         // C rows of 4096 / D
    const uint64_t *inc;
    float2 *out;
    long long out_stride, n_out;
    long long ntiles;
    long long ws0;             // window start (samples from `in`, 16-byte aligned) of row 0 of tile 0
    long long m_t0;            // output index (from this call's first) of row 0, candidate 0 of tile 0
    uint64_t n_t0;             // absolute stream index of tile 0's anchor
    int KS, Ng, Nc8, Cg, C, ngroups, stages, stage_bytes;
};

// One persistent CTA per SM, bound to one channel group; CTAs of a group stride over the tiles (groups > 1 reread the
// input, mostly from L2: the CTAs of all groups walk the tiles in the same order).
//   warps 0..2  producers: cp.async 16-byte chunks global -> SWIZZLE_64B stage (history / zeros by plain stores)
//   warp 3      MMA issuer: KS tcgen05.mma.kind::i8 per tile, M = 128 rows, N = Ng
//   warps 4..19 epilogue: (set, half, quadrant); half h converts the group's channels h, h + 2, ... of its quadrant's rows
template <int PC>
__global__ void __launch_bounds__(DDC_THREADS, 1) ddc_tc_kernel(const DdcTcArgs a) {
    constexpr int D = 32 / PC;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * DDC_STAGES + 4];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KS = a.KS, Ng = a.Ng, SB = a.stage_bytes, NST = a.stages;
    const int grp = blockIdx.x % a.ngroups;
    const long long wstride = gridDim.x / a.ngroups;
    const long long wfirst = blockIdx.x / a.ngroups;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stage0 = base;
    const uint32_t tab_s = stage0 + NST * SB;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (DDC_STAGES + s); };
    auto accf_bar = [&](int s) { return bar0 + 8u * (2 * DDC_STAGES + s); };
    auto acce_bar = [&](int s) { return bar0 + 8u * (2 * DDC_STAGES + 2 + s); };

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.tab + (size_t)grp * KS * Ng * 32);
        uint4 *dst = reinterpret_cast<uint4 *>(gen + NST * SB);
        for (int i = tid; i < KS * Ng * 2; i += DDC_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < DDC_STAGES; ++s) { mbar_init(full_bar(s), 32 * DDC_PROD_WARPS); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(accf_bar(s), 1); mbar_init(acce_bar(s), 8); }
        mbar_init_fence();
    }
    if (warp == DDC_MMA_WARP) {
        tmem_alloc<512>(smem_u32(&tmem_base_s));
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    if (warp < DDC_PROD_WARPS) {
        // ================= producers =================
        const int ptid = warp * 32 + lane;
        const int nchunks = (64 * 127 + 32 * KS + 15) / 16;
        int stage = 0;
        uint32_t ph = 0;
        for (long long t = wfirst; t < a.ntiles; t += wstride) {
            const long long w0 = a.ws0 + t * DDC_TILE;  // multiple of 8 samples from a 16-byte aligned address
            mbar_wait(empty_bar(stage), ph ^ 1u);
            const uint32_t sbase = stage0 + (uint32_t)stage * SB;
            bool slow = false;
            if (w0 >= 0 && w0 + 8LL * nchunks <= a.n_in) {
                const uint8_t *src = a.in + 2 * w0;
#pragma unroll 4
                for (int c = ptid; c < nchunks; c += 32 * DDC_PROD_WARPS) cp_async16_s(sbase + SmemLayout<64>::swz(16u * (uint32_t)c), src + 16 * c);
            } else {
                for (int c = ptid; c < nchunks; c += 32 * DDC_PROD_WARPS) {
                    const long long s0 = w0 + 8LL * c;
                    const uint32_t off = SmemLayout<64>::swz(16u * (uint32_t)c);
                    if (s0 >= 0 && s0 + 8 <= a.n_in) {
                        cp_async16_s(sbase + off, a.in + 2 * s0);
                    } else if (s0 < a.n_in) {
                        // carried history, "zero" samples (byte pair 128, 128) before the stream, or the ragged end
                        unsigned short hv[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const long long s = s0 + i;
                            unsigned short v = 0x8080;
                            if (s >= 0) { if (s < a.n_in) v = *reinterpret_cast<const unsigned short *>(a.in + 2 * s); }
                            else if (s >= -a.hist_valid) v = *reinterpret_cast<const unsigned short *>(a.hist + 2 * ((long long)a.HL + s));
                            hv[i] = v;
                        }
                        uint4 q;
                        q.x = hv[0] | ((unsigned)hv[1] << 16); q.y = hv[2] | ((unsigned)hv[3] << 16);
                        q.z = hv[4] | ((unsigned)hv[5] << 16); q.w = hv[6] | ((unsigned)hv[7] << 16);
                        *reinterpret_cast<uint4 *>(gen + (size_t)stage * SB + off) = q;
                        slow = true;
                    }
                    // chunks past the end feed only outputs that this call does not store
                }
            }
            if (slow) fence_proxy_async();
            cp_async_arrive_noinc(full_bar(stage));
            if (++stage == NST) { stage = 0; ph ^= 1u; }
        }
        cp_async_wait_all();
    } else if (warp == DDC_MMA_WARP) {
        // ================= MMA issuer =================
        const uint32_t idesc = idesc_u8s8_s32(128, Ng);
        const uint64_t bdesc0 = smem_desc(tab_s, 128, 256, 0);
        int stage = 0, as = 0;
        uint32_t ph = 0, aph = 0;
        for (long long t = wfirst; t < a.ntiles; t += wstride) {
            mbar_wait(full_bar(stage), ph);
            mbar_wait(acce_bar(as), aph ^ 1u);
            tc_fence_after();
            if (elect_one()) {
                uint64_t ad = smem_desc(stage0 + (uint32_t)stage * SB, 16, 8 * 64, SmemLayout<64>::type);
                uint64_t bd = bdesc0;
                const uint32_t d0 = tmem + (uint32_t)(as * DDC_ACC_COLS);
                umma_i8<false>(d0, ad, bd, idesc);
                for (int kk = 1; kk < KS; ++kk) {
                    ad += 2;                 // 32 bytes along the window
                    bd += (Ng * 32) >> 4;    // next tap block
                    umma_i8<true>(d0, ad, bd, idesc);
                }
                umma_commit(empty_bar(stage));
                umma_commit(accf_bar(as));
            }
            __syncwarp();
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            as ^= 1;
            if (as == 0) aph ^= 1u;
        }
    } else {
        // ================= epilogue =================
        const int ew = warp - DDC_EPI_WARP0, wg = ew >> 2, g = wg & 1, h = wg >> 1;
        const int quad = warp & 3;
        const int row = quad * 32 + lane;  // TMEM lane = window row of the tile
        const int nmine = (a.Cg - h + 1) / 2;  // channels h, h + 2, ... of the group
        const int cbase = grp * a.Cg;
        uint32_t aph = 0;
        long long it = 0;
        for (long long t = wfirst; t < a.ntiles; t += wstride, ++it) {
            if ((it & 1) != g) continue;
            // tile anchors: one exact sincospi per channel, lane i for this warp's i-th channel
            float2 bl = make_float2(1.f, 0.f);
            {
                const int c = cbase + h + 2 * lane;
                if (lane < nmine && c < a.C) bl = nco_rot((a.n_t0 + (uint64_t)(t * DDC_TILE)) * __ldg(a.inc + c));
            }
            const long long m_row = a.m_t0 + t * (DDC_TILE / D) + (long long)row * PC;  // output of candidate 0
            mbar_wait(accf_bar(g), aph);
            aph ^= 1u;
            tc_fence_after();
            const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(g * DDC_ACC_COLS);
            for (int i = 0; i < nmine; ++i) {
                const int cl = h + 2 * i, c = cbase + cl;
                const float2 b = make_float2(__shfl_sync(0xffffffffu, bl.x, i), __shfl_sync(0xffffffffu, bl.y, i));
                if (c >= a.C) break;  // uniform: padding channels of the last group
                const DdcChan k = a.chan[c];
                const float2 *rt = a.rot + (size_t)c * (DDC_TILE / D) + row * PC;
                float2 *out = a.out + (long long)c * a.out_stride;
                const uint32_t col0 = tbase + (uint32_t)(cl * a.Nc8);
                constexpr int CU = PC < 4 ? PC : 4;  // candidates per TMEM load round
#pragma unroll
                for (int k0 = 0; k0 < PC; k0 += CU) {
                    // v[dg * 2CU + 2u + part] = digit dg of part (I / Q) of candidate k0 + u
                    uint32_t v[24];
                    if constexpr (PC <= 2) {
                        // the channel's 8 (PC = 1) or 16 (PC = 2) columns hold (dg, u, part) at dg * 2 PC + 2u + part
                        tmem_ld_32x32b_x8(col0, v);
                        if constexpr (PC == 2) tmem_ld_32x32b_x8(col0 + 8, v + 8);
                    } else {
#pragma unroll
                        for (int dg = 0; dg < 3; ++dg) tmem_ld_32x32b_x8(col0 + dg * 2 * PC + 2 * k0, v + 8 * dg);
                    }
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < CU; ++u) {
                        const long long m = m_row + k0 + u;
                        const int i0 = 2 * u;
                        constexpr int DS = PC <= 2 ? 2 * PC : 8;  // register distance between digits
                        const float fI = (float)((int)(v[DS + i0] << 8) + (int)v[i0] + k.c10[0]);
                        const float fQ = (float)((int)(v[DS + i0 + 1] << 8) + (int)v[i0 + 1] + k.c10[1]);
                        const float gI = __int_as_float((int)v[2 * DS + i0] + k.m2[0]) - 12582912.0f;
                        const float gQ = __int_as_float((int)v[2 * DS + i0 + 1] + k.m2[1]) - 12582912.0f;
                        const float2 z = make_float2(fmaf(gI, k.sc2, fI * k.sc0), fmaf(gQ, k.sc2, fQ * k.sc0));
                        const float2 r = cmul(b, __ldg(rt + k0 + u));
                        if (m >= 0 && m < a.n_out) out[m] = cmul(r, z);
                    }
                }
            }
            // the set is read: hand it back to the MMA warp (8 warps arrive)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acce_bar(g));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == DDC_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

// Where the samples of one call live: s < 0 is the carried history (hist[HL + s], the last hist_valid of them belong to
// the stream, older ones read as zero), 0 <= s < n_in the caller's block.
struct DdcSrc {
    const void *in, *hist;
    long long n_in, hist_valid;
    int HL;
};

template <bool U8>
__device__ __forceinline__ float2 ddc_load(const DdcSrc &s, long long i) {
    if (i < -s.hist_valid) return make_float2(0.f, 0.f);
    const bool hh = i < 0;
    const void *base = hh ? s.hist : s.in;
    const long long k = hh ? i + s.HL : i;
    if (U8) return unpack_iq_u16(__ldg(reinterpret_cast<const uint16_t *>(base) + k));
    return __ldg(reinterpret_cast<const float2 *>(base) + k);
}

constexpr int DDC_GEN_CB = 8;  // channels per thread of the general kernel

// One thread per (output, block of 8 channels).  Output m's newest sample is s = s0 + m D (from `in`), absolute index
// n0 + m D.  Taps g: C rows of L complex.
template <bool U8>
__global__ void __launch_bounds__(256) ddc_general_kernel(DdcSrc src, const float2 *__restrict__ g, int L, int C,
                                                          long long D, long long s0, uint64_t n0,
                                                          const uint64_t *__restrict__ inc, long long n_out,
                                                          float2 *__restrict__ out, long long out_stride) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int c0 = blockIdx.y * DDC_GEN_CB;
    if (m >= n_out) return;
    const int nc = min(DDC_GEN_CB, C - c0);
    float ar[DDC_GEN_CB], ai[DDC_GEN_CB];
#pragma unroll
    for (int c = 0; c < DDC_GEN_CB; ++c) ar[c] = ai[c] = 0.f;
    const long long e = s0 + m * D;
    for (int j = 0; j < L; ++j) {
        const float2 x = ddc_load<U8>(src, e - j);
#pragma unroll
        for (int c = 0; c < DDC_GEN_CB; ++c) {
            if (c < nc) {
                const float2 t = __ldg(g + (size_t)(c0 + c) * L + j);
                ar[c] = __fmaf_rn(t.x, x.x, ar[c]);
                ar[c] = __fmaf_rn(-t.y, x.y, ar[c]);
                ai[c] = __fmaf_rn(t.x, x.y, ai[c]);
                ai[c] = __fmaf_rn(t.y, x.x, ai[c]);
            }
        }
    }
    const uint64_t n = n0 + (uint64_t)(m * D);
#pragma unroll
    for (int c = 0; c < DDC_GEN_CB; ++c)
        if (c < nc) out[(long long)(c0 + c) * out_stride + m] = cmul(nco_rot(n * __ldg(inc + c0 + c)), make_float2(ar[c], ai[c]));
}

}  // namespace

extern "C" uint64_t sdr_ddc_phase_increment(double freq, double rate) {
    if (!std::isfinite(freq) || !std::isfinite(rate) || rate == 0.0) return 0;
    double nu = freq / rate;
    if (!std::isfinite(nu)) return 0;
    nu -= std::round(nu);  // exact: |nu| <= 0.5
    if (std::fabs(nu) == 0.5) return (uint64_t)1 << 63;
    return (uint64_t)std::llround(std::ldexp(nu, 64));  // |nu 2^64| <= 2^63 - 2^10: fits, negative = two's complement
}

struct DdcHost {
    int dev = 0;
    size_t L = 0, C = 0, D = 1, HL = 0, n_sets = 1;
    uint64_t first = 0;
    int fmt = SDR_FMT_U8IQ;
    unsigned flags = 0;
    std::vector<float> taps;   // n_sets x L, as given
    std::vector<uint64_t> inc;
    // tensor path geometry (tc = false: general kernel)
    bool tc = false;
    int PC = 0, KS = 0, Nc8 = 0, Cg = 0, ngroups = 0, Ng = 0, stages = 0;
    size_t smem = 0;
    long long total = 0;       // input samples seen
    int last_path = 0;
};

static size_t ddc_es(const DdcHost *h) { return h->fmt == SDR_FMT_U8IQ ? 2 : 8; }

struct sdr_ddc : DdcHost {
    StreamRef stream;
    DevBuf d_tab, d_chan, d_rot, d_g, d_inc;
    DevBuf d_hist[2];          // the last HL inputs before `total`, raw format
    int cur = 0;
    DevBuf d_in, d_out;

    int alloc(void *user_stream, const sdr_ddc *);
    int copy_device(const sdr_ddc &src) {
        if (HL == 0) return SDR_OK;
        return cuda_status(cudaMemcpy(d_hist[0].p, src.d_hist[src.cur].p, HL * ddc_es(this), cudaMemcpyDeviceToDevice));
    }
};

// Tensor-path geometry: D | 32, rows 32 samples apart, PC = 32 / D candidates per row and channel (all kept), a channel's
// 6 PC columns padded to Nc8 (a multiple of 8), Cg channels per group with Ng = Cg Nc8 rounded up to 16 <= 256 columns
// (two accumulator sets in TMEM) and the group's table plus >= 2 stages in shared memory.  False: the general kernel.
static bool ddc_tc_geometry(DdcHost *h) {
    if (h->fmt != SDR_FMT_U8IQ || (h->flags & SDR_DDC_GENERAL_KERNEL) || h->D > 32 || 32 % h->D != 0 ||
        h->L > (size_t)DDC_MAX_TC_K)
        return false;
    const int PC = 32 / (int)h->D, KS = fir_umma_ksteps((int)h->L, 32, PC);
    const int Nc8 = (6 * PC + 7) / 8 * 8;
    int cmax = 0;
    for (int c = 1; c <= (int)h->C && c * Nc8 <= DDC_ACC_COLS; ++c) {
        const int Ng = (c * Nc8 + 15) / 16 * 16;
        if (ddc_smem_bytes(KS, Ng, 2) > DDC_SMEM_MAX) break;
        cmax = c;
    }
    if (!cmax) return false;
    const int ngroups = ((int)h->C + cmax - 1) / cmax;
    h->Cg = ((int)h->C + ngroups - 1) / ngroups;  // balanced groups
    h->ngroups = ngroups;
    h->Ng = (h->Cg * Nc8 + 15) / 16 * 16;
    h->PC = PC; h->KS = KS; h->Nc8 = Nc8;
    int st = DDC_STAGES;
    while (st > 2 && ddc_smem_bytes(KS, h->Ng, st) > DDC_SMEM_MAX) --st;
    h->stages = st;
    h->smem = ddc_smem_bytes(KS, h->Ng, st);
    return true;
}

// complex taps g_k[j] = h_k[j] e^{+2 pi i (j Delta_k mod 2^64) / 2^64}, rounded to f32 from f64
static void ddc_rotated_taps(const DdcHost *h, size_t k, std::vector<float> &g) {
    nco_rotated_taps(h->taps.data() + (h->n_sets == 1 ? 0 : k * h->L), h->L, h->inc[k], g);
}

// tables, taps and history buffers of a handle whose configuration fields are set
int sdr_ddc::alloc(void *user_stream, const sdr_ddc *) {
    int rc = stream.init(user_stream);
    if (rc) return rc;
    cudaStream_t st = stream.s;
    tc = ddc_tc_geometry(this);
    std::vector<float> g;
    if (tc) {
        // group tables [delta][group][kk][Ng x 32 B canonical K-major block]; channel cl of a group owns columns
        // cl Nc8 + dg 2PC + 2u + part.  D = 16, 32 take the PC = 4 tables (whose 6 PC column count is a whole number of
        // core matrices) and keep every (8 / PC)-th candidate; their first KS k-steps hold all the kept candidates' taps.
        const int PCb = std::max(PC, 4), sig = PCb / PC;
        const size_t blk = (size_t)Ng * 32, grp_bytes = (size_t)KS * blk;
        std::vector<uint8_t> tab((size_t)8 * ngroups * grp_bytes, 0), one;
        std::vector<DdcChan> chan(C);
        const int TR = DDC_TILE / (int)D;
        std::vector<float> rot(2 * C * TR);
        for (size_t k = 0; k < C; ++k) {
            ddc_rotated_taps(this, k, g);
            int magic[2][3];
            float sc[3];
            if (!fir_umma_build_tables(g.data(), (int)L, true, 32, PCb, 0, (int)D, one, magic, sc)) return SDR_ERR_INVALID_ARG;
            const int KSb = fir_umma_ksteps((int)L, 32, PCb), Nb = 6 * PCb;
            const size_t grp = k / Cg, cl = k % Cg;
            for (int delta = 0; delta < 8; ++delta)
                for (int kk = 0; kk < KS; ++kk) {
                    const uint8_t *sb = one.data() + ((size_t)delta * KSb + kk) * Nb * 32;
                    uint8_t *db = tab.data() + ((size_t)delta * ngroups + grp) * grp_bytes + (size_t)kk * blk;
                    for (int dg = 0; dg < 3; ++dg)
                        for (int u = 0; u < PC; ++u)
                            for (int part = 0; part < 2; ++part) {
                                const int ns = dg * 2 * PCb + 2 * sig * u + part;
                                const int nd = (int)cl * Nc8 + dg * 2 * PC + 2 * u + part;
                                for (int kb = 0; kb < 32; ++kb) {
                                    const int o = (kb / 16) * 128 + kb % 16;
                                    db[(nd / 8) * 256 + (nd % 8) * 16 + o] = sb[(ns / 8) * 256 + (ns % 8) * 16 + o];
                                }
                            }
                }
            chan[k] = DdcChan{{magic[0][0], magic[1][0]}, {magic[0][2], magic[1][2]}, sc[0], sc[2]};
            for (int j = 0; j < TR; ++j) {
                const double t = NCO_2PI * nco_turns(((uint64_t)D * j + D - 1) * inc[k]);
                rot[2 * (k * TR + j)] = (float)std::cos(t);
                rot[2 * (k * TR + j) + 1] = (float)-std::sin(t);
            }
        }
        if ((rc = d_tab.upload(tab.data(), tab.size(), st))) return rc;
        if ((rc = d_chan.upload(chan.data(), chan.size() * sizeof(DdcChan), st))) return rc;
        if ((rc = d_rot.upload(rot.data(), rot.size() * sizeof(float), st))) return rc;
    } else {
        std::vector<float> all(2 * C * L);
        for (size_t k = 0; k < C; ++k) {
            ddc_rotated_taps(this, k, g);
            std::copy(g.begin(), g.end(), all.begin() + 2 * k * L);
        }
        if ((rc = d_g.upload(all.data(), all.size() * sizeof(float), st))) return rc;
    }
    if ((rc = d_inc.upload(inc.data(), C * sizeof(uint64_t), st))) return rc;
    for (int i = 0; i < 2; ++i)
        if ((rc = d_hist[i].reserve(std::max<size_t>(HL, 2) * ddc_es(this)))) return rc;
    return cuda_status(cudaStreamSynchronize(st));
}

extern "C" sdr_ddc_t *sdr_ddc_create(const sdr_ddc_config_t *cfg, int *err) {
    if (!cfg || !cfg->taps || !cfg->phase_inc || cfg->n_taps == 0 || cfg->n_taps > ((size_t)1 << 20) ||
        cfg->n_channels == 0 || cfg->n_channels > DDC_MAX_CH ||
        (cfg->n_tap_sets != 1 && cfg->n_tap_sets != cfg->n_channels) || cfg->decimation == 0 ||
        cfg->decimation > ((size_t)1 << 40) || (cfg->input_format != SDR_FMT_U8IQ && cfg->input_format != SDR_FMT_C64) ||
        (cfg->flags & ~SDR_DDC_GENERAL_KERNEL))
        return fail(err, SDR_ERR_INVALID_ARG);
    for (size_t i = 0; i < cfg->n_taps * cfg->n_tap_sets; ++i)
        if (!std::isfinite(cfg->taps[i])) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_ddc>(err, cfg->device, cfg->stream, [&](sdr_ddc &h) {
        h.L = cfg->n_taps;
        h.C = cfg->n_channels;
        h.D = cfg->decimation;
        h.HL = h.L - 1;
        h.n_sets = cfg->n_tap_sets;
        h.first = cfg->first_sample;
        h.fmt = cfg->input_format;
        h.flags = cfg->flags;
        h.taps.assign(cfg->taps, cfg->taps + h.L * h.n_sets);
        h.inc.assign(cfg->phase_inc, cfg->phase_inc + h.C);
        return SDR_OK;
    });
}

extern "C" void sdr_ddc_destroy(sdr_ddc_t *h) { destroy_handle(h); }

extern "C" int sdr_ddc_reset(sdr_ddc_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    // history older than the stream reads as zero (hist_valid = min(HL, total)), so the stale buffer is never used
    h->total = 0;
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_ddc_t *sdr_ddc_clone(const sdr_ddc_t *src, int *err) { return clone_handle<DdcHost>(src, err); }

extern "C" size_t sdr_ddc_output_count(const sdr_ddc_t *h, size_t n_in) {
    if (!h) return 0;
    const long long D = (long long)h->D;
    return (size_t)((h->total + (long long)n_in) / D - h->total / D);
}

extern "C" int sdr_ddc_last_path(const sdr_ddc_t *h) { return h ? h->last_path : 0; }

static int ddc_launch_tc(sdr_ddc *h, const void *in, size_t n_in, float2 *out, size_t out_stride, size_t nf) {
    const long long D = (long long)h->D, L = (long long)h->L, total = h->total;
    // tile anchors sit at absolute N = eps (mod 4096), eps = F mod D; in handle coordinates i = N - F at i = -off (mod 4096)
    const long long off = (long long)((h->first - h->first % h->D) % DDC_TILE);
    const long long m0 = total / D;
    const long long i_first = D * m0 + D - 1, i_last = D * (m0 + (long long)nf - 1) + D - 1;
    const long long T0 = (i_first + off) / DDC_TILE, T1 = (i_last + off) / DDC_TILE;
    DdcTcArgs a;
    a.in = (const uint8_t *)in;
    a.hist = (const uint8_t *)h->d_hist[h->cur].p;
    a.n_in = (long long)n_in;
    a.hist_valid = std::min<long long>((long long)h->HL, total);
    a.HL = (int)h->HL;
    const long long tile0_s = T0 * DDC_TILE - off - total;  // tile 0's anchor, samples from `in`
    long long delta = ((long long)(((uintptr_t)in & 15) >> 1) + tile0_s + D - L) % 8;
    if (delta < 0) delta += 8;
    a.ws0 = tile0_s + D - 1 - (L - 1) - delta;
    a.tab = (const uint8_t *)h->d_tab.p + (size_t)delta * h->ngroups * h->KS * h->Ng * 32;
    a.chan = (const DdcChan *)h->d_chan.p;
    a.rot = (const float2 *)h->d_rot.p;
    a.inc = (const uint64_t *)h->d_inc.p;
    a.out = out;
    a.out_stride = (long long)out_stride;
    a.n_out = (long long)nf;
    a.ntiles = T1 - T0 + 1;
    a.m_t0 = (T0 * DDC_TILE - off) / D - m0;
    a.n_t0 = h->first + (uint64_t)(T0 * DDC_TILE - off);
    a.KS = h->KS; a.Ng = h->Ng; a.Nc8 = h->Nc8; a.Cg = h->Cg; a.C = (int)h->C; a.ngroups = h->ngroups;
    a.stages = h->stages;
    a.stage_bytes = ddc_stage_bytes(h->KS);
    const long long per = std::max<long long>(1, std::min<long long>(a.ntiles, current_sm_count() / h->ngroups));
    const unsigned grid = (unsigned)(per * h->ngroups);
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem);
        if (e != cudaSuccess) return cuda_status(e);
        kern<<<grid, DDC_THREADS, h->smem, h->stream.s>>>(a);
        count_launch();
        return launch_status();
    };
    switch (h->PC) {
        case 1: return go(ddc_tc_kernel<1>);
        case 2: return go(ddc_tc_kernel<2>);
        case 4: return go(ddc_tc_kernel<4>);
        case 8: return go(ddc_tc_kernel<8>);
        case 16: return go(ddc_tc_kernel<16>);
        case 32: return go(ddc_tc_kernel<32>);
    }
    return SDR_ERR_UNSUPPORTED;
}

static int ddc_launch_general(sdr_ddc *h, const void *in, size_t n_in, float2 *out, size_t out_stride, size_t nf) {
    const long long D = (long long)h->D, total = h->total, m0 = total / D;
    DdcSrc s;
    s.in = in;
    s.hist = h->d_hist[h->cur].p;
    s.n_in = (long long)n_in;
    s.hist_valid = std::min<long long>((long long)h->HL, total);
    s.HL = (int)h->HL;
    const long long i0 = D * m0 + D - 1;  // newest sample of this call's first output (handle coordinates)
    const dim3 grid((unsigned)(((long long)nf + 255) / 256), (unsigned)((h->C + DDC_GEN_CB - 1) / DDC_GEN_CB));
    const uint64_t n0 = h->first + (uint64_t)i0;
    if (h->fmt == SDR_FMT_U8IQ)
        ddc_general_kernel<true><<<grid, 256, 0, h->stream.s>>>(s, (const float2 *)h->d_g.p, (int)h->L, (int)h->C, D,
                                                                i0 - total, n0, (const uint64_t *)h->d_inc.p,
                                                                (long long)nf, out, (long long)out_stride);
    else
        ddc_general_kernel<false><<<grid, 256, 0, h->stream.s>>>(s, (const float2 *)h->d_g.p, (int)h->L, (int)h->C, D,
                                                                 i0 - total, n0, (const uint64_t *)h->d_inc.p,
                                                                 (long long)nf, out, (long long)out_stride);
    count_launch();
    return launch_status();
}

// in: n_in device samples; out: C rows of out_stride, nf outputs each
static int ddc_run(sdr_ddc *h, const void *in, size_t n_in, float *out, size_t out_stride, size_t nf) {
    cudaStream_t st = h->stream.s;
    const size_t es = ddc_es(h);
    if (nf > 0) {
        const int rc = h->tc ? ddc_launch_tc(h, in, n_in, (float2 *)out, out_stride, nf)
                             : ddc_launch_general(h, in, n_in, (float2 *)out, out_stride, nf);
        if (rc) return rc;
        h->last_path = h->tc ? 2 : 1;
    }
    // history = the last HL samples of (history, input)
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

static int ddc_check(const sdr_ddc *h, const void *in, size_t n_in, const float *out, size_t out_cap,
                     size_t out_stride, size_t *n_out, size_t *nf) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out) return SDR_ERR_BAD_DATA_PTR;
    *n_out = 0;
    if (n_in > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    *nf = sdr_ddc_output_count(h, n_in);
    if (*nf > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (*nf > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (*nf > 0 && out_stride < *nf) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_ddc_process_dev(sdr_ddc_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                                   size_t out_stride, size_t *n_out) {
    size_t nf = 0;
    int rc = ddc_check(h, in, n_in, out_c64, out_cap, out_stride, n_out, &nf);
    if (rc) return rc;
    if (((uintptr_t)in % ddc_es(h)) != 0 || ((uintptr_t)out_c64 % 8) != 0) return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    rc = ddc_run(h, in, n_in, out_c64, out_stride, nf);
    if (rc) return rc;
    *n_out = nf;
    return SDR_OK;
}

extern "C" int sdr_ddc_process(sdr_ddc_t *h, const void *in, size_t n_in, float *out_c64, size_t out_cap,
                               size_t out_stride, size_t *n_out) {
    size_t nf = 0;
    int rc = ddc_check(h, in, n_in, out_c64, out_cap, out_stride, n_out, &nf);
    if (rc) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t es = ddc_es(h), D = h->D, C = h->C;
    cudaStream_t st = h->stream.s;
    // chunks of at most ~32 MiB of input and of output: H2D, compute, D2H in stream order
    size_t chunk = std::max<size_t>(1, DDC_SLAB_BYTES / es);
    chunk = std::max<size_t>(1, std::min(chunk, (DDC_SLAB_BYTES / (8 * C) + 1) * D));
    chunk = std::min(chunk, std::max<size_t>(n_in, 1));
    const size_t fcap = chunk / D + 1;
    rc = h->d_in.reserve(chunk * es);
    if (!rc) rc = h->d_out.reserve(fcap * C * 8);
    if (rc) return rc;
    size_t done_in = 0, done_out = 0;
    while (done_in < n_in) {
        const size_t cnt = std::min(chunk, n_in - done_in);
        const size_t cnf = sdr_ddc_output_count(h, cnt);
        SDR_CUDA_TRY(cudaMemcpyAsync(h->d_in.p, (const char *)in + done_in * es, cnt * es, cudaMemcpyHostToDevice, st));
        rc = ddc_run(h, h->d_in.p, cnt, (float *)h->d_out.p, fcap, cnf);
        if (rc) return rc;
        if (cnf > 0)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(out_c64 + done_out * 2, out_stride * 8, h->d_out.p, fcap * 8, cnf * 8, C,
                                           cudaMemcpyDeviceToHost, st));
        done_in += cnt;
        done_out += cnf;
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    *n_out = done_out;
    return SDR_OK;
}

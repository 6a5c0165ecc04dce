// fir_umma_c64.cu -- K5c: Fir<f32, Complex<f32>> on a Complex<f32> (c64) stream, many channels, on the 5th-generation
// tensor cores (tcgen05 / TMEM).  This is the north star's "large-batch multi-channel FIR recast as a dense Toeplitz
// GEMM": config C4's 1024 channel streams x 255 real taps (examples/pll.rs front end), which the CUDA-core kernel
// (fir.cu, 2 K FMA per sample) runs FP32-pipe bound at ~12 % of its HBM roofline.
//
// Reference functions: signal::Filter::next -> Fir::apply (src/signal/adapters/mod.rs:94-96, src/filter/fir.rs:23-32),
// Convolve for Complex<f32> * f32 (src/filter/convolve.rs:13-15): y[n] = sum_k c[k] x[n-k], re and im independently.
//
// Arithmetic.  f32 samples and taps are split into bf16 terms with round-to-nearest, x = xh + xm (+ xl), c = ch + cm
// (+ cl); every bf16 x bf16 product is exact in the tensor core's f32 accumulator.  NS = 3 keeps the six products down
// to 2^-16 (hh, hm, mh, hl, mm, lh): the result carries the split's residual 2^-24 relative and the f32 accumulation,
// i.e. the reference's own accuracy (measured 3e-7 of max|y| vs the f64 truth, reference order 6e-7).  NS = 2
// (SDR_FIR_SPLIT2) keeps three products (hh, hm, mh): 2^-18-grade terms are dropped, 4-5e-6 of max|y| on noise -- inside
// the north star's 1e-5, 1.5x less tensor work.  Non-finite samples poison the whole row window (a Toeplitz zero times
// Inf is NaN); callers that need Fir::apply's exact non-finite behaviour use SDR_FIR_STRICT_ORDER.
//
// Data flow of a 4096-output tile (one channel, 128 window rows x 32 outputs):
//   * TMA: ONE cp.async.bulk (UBLKCP) brings the tile's raw c64 window (4096 + K - 1 samples + k-step padding, ~35 KB)
//     from HBM into a raw ring slot, completion on an mbarrier (complete_tx).  Tiles that touch the start of the
//     stream (carried history / zeros, fir.rs:15) or its ragged end are filled by plain loads instead.
//   * 8 producer warps split the raw slot into 2 NS bf16 PLANES (re / im x h, m[, l]): 8 samples per lane and step,
//     4 LDS.128 -> cvt.rn.bf16x2 / subtract -> one 16-byte chunk per plane, stored with the SWIZZLE_64B XOR.
//   * A operand = a plane read through a shared-memory matrix descriptor whose 128 rows OVERLAP (row pitch 64 B = 32
//     samples inside one flat plane; the swizzle XOR is a function of the absolute address, so overlapping rows agree:
//     scripts/probes/umma_toeplitz_probe.cu).  B operand = banded Toeplitz block of the bf16 tap terms, columns
//     [ch | cm | cl] x 32 outputs.  Per k-step (16 samples) and part: MMA(xh, N = 32 NS), MMA(xm, N = 32 (NS-1)),
//     [MMA(xl, N = 32)] accumulate Sh | Sm | Sl in TMEM (f32); y = Sh + Sm + Sl in the epilogue.
//   * 16 epilogue warps (2 accumulator sets x 2 column halves): tcgen05.ld.16x256b fragments give every thread two
//     adjacent outputs of two rows for re and im -> one 16-byte store of (re, im, re, im); 4 threads = one 64-byte run.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_bf16.h>

#include "kernels.h"
#include "ptx.cuh"

namespace sdr {

namespace {

constexpr int UC_P = 32;                 // outputs per window row (row pitch 64 B of bf16: SWIZZLE_64B)
constexpr int UC_ROWS = 128;             // window rows per tile = MMA M
constexpr int UC_TILE = UC_P * UC_ROWS;  // outputs per tile
constexpr int UC_PROD_WARPS = 8;
constexpr int UC_MMA_WARP = UC_PROD_WARPS;
constexpr int UC_EPI_WARP0 = UC_PROD_WARPS + 1;
constexpr int UC_THREADS = (UC_PROD_WARPS + 1 + 16) * 32;
constexpr int UC_MAX_STAGES = 3;
constexpr int UC_RAW = 2;                // raw ring slots (one when shared memory is short: 255 taps x 3 terms)
constexpr int UC_MAX_K = 511;

struct UcArgs {
    FirArgs f;
    const uint8_t *tab;  // this call's alignment variant: KS blocks of (32 NS) x 32 bytes, canonical no-swizzle K-major
    int KS;              // k-steps of 16 samples
    int delta;           // the first needed sample sits `delta` (0 / 1) elements into the plane (16-byte raw alignment)
    int ntiles;          // tiles per channel
    int nel;             // plane elements (= raw samples) a tile uses: 127 * 32 + 16 KS, a multiple of 16
    int plane_bytes;     // 2 * nel rounded up to 1024 (swizzle period)
    int stages;
    int nraw;            // raw ring slots: 2 = the next tile's window lands while this one is converted, 1 = after it
    // per-channel taps (the polyphase branches of the rational resampler): channel c filters with the table at
    // tab + c * tab_stride, and every CTA is bound to ONE channel (c = blockIdx.x mod n_ch) so that it loads one table
    long long tab_stride; // 0 = all channels share `tab`
};

__device__ __forceinline__ void prod_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(UC_PROD_WARPS * 32) : "memory"); }

// split 8 f32 values (4 pairs; pair i belongs to word (i + rot) & 3 of the 16-byte chunk) into bf16 terms, round to
// nearest even, and store one 4-byte word per pair and term
template <int NS>
__device__ __forceinline__ void split_store(const float (&v)[8], uint8_t *plane0, int plane_bytes, uint32_t off, int rot) {
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = v[i];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 b = __floats2bfloat162_rn(r[2 * i], r[2 * i + 1]);  // .x = low half = the even element
            const uint32_t w = *reinterpret_cast<const uint32_t *>(&b);
            if (s + 1 < NS) {
                r[2 * i] = __fsub_rn(r[2 * i], __uint_as_float(w << 16));
                r[2 * i + 1] = __fsub_rn(r[2 * i + 1], __uint_as_float(w & 0xFFFF0000u));
            }
            *reinterpret_cast<uint32_t *>(plane0 + (size_t)s * plane_bytes + off + 4u * (uint32_t)((i + rot) & 3)) = w;
        }
    }
}

__host__ __device__ constexpr int uc_ksteps(int K) { return (K - 1 + 1 + UC_P + 15) / 16; }  // K-1 taps back, delta <= 1, 32 outputs
__host__ __device__ constexpr int uc_nel(int KS) { return (UC_ROWS - 1) * UC_P + 16 * KS; }
__host__ __device__ constexpr int uc_plane_bytes(int KS) { return (2 * uc_nel(KS) + 1023) / 1024 * 1024; }
__host__ __device__ constexpr size_t uc_smem_bytes(int NS, int KS, int stages, int nraw) {
    // stages of 2 NS planes + tap tables + raw ring + 1 KB alignment slack
    return (size_t)stages * 2 * NS * uc_plane_bytes(KS) + (size_t)KS * 32 * NS * 32 + (size_t)nraw * 8 * uc_nel(KS) + 1024;
}
constexpr size_t UC_SMEM_MAX = 225 * 1024;
// the roomiest configuration that fits: prefer a second raw slot, then a third plane stage
inline bool uc_pick(int NS, int KS, int *stages, int *nraw) {
    static const int pref[4][2] = {{3, 2}, {2, 2}, {3, 1}, {2, 1}};
    for (auto &p : pref)
        if (uc_smem_bytes(NS, KS, p[0], p[1]) <= UC_SMEM_MAX) { *stages = p[0]; *nraw = p[1]; return true; }
    return false;
}

template <int NS>
__global__ void __launch_bounds__(UC_THREADS, 1) fir_umma_c64_kernel(const UcArgs a) {
    constexpr int NCOL = 32 * NS;       // table columns = accumulator columns per part
    constexpr int SETC = 2 * NCOL;      // TMEM columns per accumulator set (re block, im block)
    constexpr int TMEM_COLS = (2 * SETC <= 256) ? 256 : 512;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * UC_MAX_STAGES + 4 + UC_RAW];
    __shared__ uint32_t tmem_base_s;
    const FirArgs &f = a.f;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KS = a.KS, NST = a.stages, PB = a.plane_bytes, SB = 2 * NS * PB, NEL = a.nel;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stage0 = base;
    const uint32_t tab_s = stage0 + NST * SB;
    const uint32_t raw_s = tab_s + KS * NCOL * 32;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));
    uint8_t *raw_g = gen + (size_t)NST * SB + (size_t)KS * NCOL * 32;
    const int RAWB = 8 * NEL;
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (UC_MAX_STAGES + s); };
    auto accf_bar = [&](int s) { return bar0 + 8u * (2 * UC_MAX_STAGES + s); };
    auto acce_bar = [&](int s) { return bar0 + 8u * (2 * UC_MAX_STAGES + 2 + s); };
    auto raw_bar = [&](int s) { return bar0 + 8u * (2 * UC_MAX_STAGES + 4 + s); };

    // work items.  Shared taps: item w = ch * ntiles + tile, CTA b takes w = b, b + grid, ...  Per-channel taps: CTA b is
    // bound to channel b mod n_ch and takes that channel's tiles i, i + cpc, ... (i = b div n_ch, cpc = CTAs on the channel)
    const bool bound = a.tab_stride != 0;
    const int my_ch = bound ? (int)(blockIdx.x % f.n_ch) : -1;
    const long long w_begin = bound ? (long long)(blockIdx.x / f.n_ch) : (long long)blockIdx.x;
    const long long w_step = bound ? (long long)((gridDim.x - my_ch + f.n_ch - 1) / f.n_ch) : (long long)gridDim.x;
    const long long w_end = bound ? (long long)a.ntiles : (long long)a.ntiles * f.n_ch;
    // ---- one-time setup ----
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.tab + (bound ? (long long)my_ch * a.tab_stride : 0LL));
        uint4 *dst = reinterpret_cast<uint4 *>(gen + (size_t)NST * SB);
        for (int i = tid; i < KS * NCOL * 2; i += UC_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < UC_MAX_STAGES; ++s) { mbar_init(full_bar(s), 32 * UC_PROD_WARPS); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(accf_bar(s), 1); mbar_init(acce_bar(s), 8); }
        for (int s = 0; s < UC_RAW; ++s) mbar_init(raw_bar(s), 1);
        mbar_init_fence();
    }
    if (warp == UC_MMA_WARP) {
        tmem_alloc<TMEM_COLS>(smem_u32(&tmem_base_s));
    }
    fence_proxy_async();  // the tap tables were written through the generic proxy, tcgen05.mma reads through the async one
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    const long long nwork = w_end;
    const long long wstride = w_step;
    // first raw sample of tile wt (in the channel's input coordinates): 16-byte aligned address by choice of delta
    auto tile_s0 = [&](long long wt) { return wt * (long long)UC_TILE - (f.K - 1) - a.delta; };
    // (a 64-bit division is ~100 instructions, and every role splits its work index several times per tile: ncu put 10 % of
    // the producers' samples on it at 1024 channels)
    // MEASURED AND REMOVED (round 2): with ONE raw slot, refilling it in two parts (the first 2048 elements are dead behind
    // the conversion's first pass) so that the next tile's copy starts half a conversion earlier: 134 vs 145 Gsamples/s on
    // one box at 255 taps (two smaller bulk copies and one more producer barrier per tile cost more than the overlap gives).
    const bool nwork32 = w_end <= 0x7fffffffLL;
    auto split = [&](long long w, int &ch, long long &wt) {
        if (bound) { ch = my_ch; wt = w; }
        else if (f.n_ch == 1) { ch = 0; wt = w; }
        else if (nwork32) { const unsigned c = (unsigned)w / (unsigned)a.ntiles; ch = (int)c; wt = (long long)((unsigned)w - c * (unsigned)a.ntiles); }
        else { ch = (int)(w / a.ntiles); wt = w - (long long)ch * a.ntiles; }
    };

    if (warp < UC_PROD_WARPS) {
        // ================= producers =================
        const int ptid = warp * 32 + lane;
        // Elements [e_lo, e_hi) of a tile's window are real input samples at 16-byte aligned addresses: ONE bulk copy.
        // What is left -- carried history / zeros in front of the stream (fir.rs:15), zeros behind its end, at most one
        // odd sample at either side -- is a few hundred elements of the first and last tile of a channel: plain stores.
        const bool gather = f.in_step != 0;
        auto tma_range = [&](long long w, int &e_lo, int &e_hi) {
            e_lo = e_hi = 0;
            if (w >= nwork || gather) return;
            int ch; long long wt;
            split(w, ch, wt);
            const long long s0 = tile_s0(wt);
            long long lo = s0 < 0 ? -s0 : 0, hi = f.n_in - s0;
            if (hi > NEL) hi = NEL;
            lo = (lo + 1) & ~1LL;
            hi &= ~1LL;
            if (hi > lo) { e_lo = (int)lo; e_hi = (int)hi; }
        };
        auto issue_tma = [&](long long w, int slot) {   // one elected thread
            int e_lo, e_hi;
            tma_range(w, e_lo, e_hi);
            if (e_hi <= e_lo) return;
            int ch; long long wt;
            split(w, ch, wt);
            const float2 *src = (const float2 *)f.in + (long long)ch * f.in_stride + tile_s0(wt) + e_lo;
            const uint32_t bytes = 8u * (uint32_t)(e_hi - e_lo);
            mbar_arrive_expect_tx(raw_bar(slot), bytes);
            tma_bulk_g2s(raw_s + (uint32_t)slot * RAWB + 8u * (uint32_t)e_lo, src, bytes, raw_bar(slot));
        };
        if (ptid == 0) issue_tma(w_begin, 0);
        const bool two = a.nraw == 2;
        int stage = 0, slot = 0;
        uint32_t ph = 0, rph[UC_RAW] = {0, 0};
        for (long long w = w_begin; w < nwork; w += wstride) {
            // the next tile's window goes into the other slot (last read one iteration ago, before the closing barrier)
            if (two && ptid == 0) issue_tma(w + wstride, slot ^ 1);
            uint8_t *rs = raw_g + (size_t)slot * RAWB;
            int e_lo, e_hi;
            tma_range(w, e_lo, e_hi);
            if (gather) {
                // polyphase branch of the resampler: the window is a strided view of the caller's frames (every in_step-th
                // frame from in_off - ch), zero outside them.  8-byte loads at a 8 in_step-byte stride: the other
                // branches' CTAs read the neighbouring frames of the same sectors, so HBM still sees every frame once
                int ch; long long wt;
                split(w, ch, wt);
                const long long j0 = f.in_step * tile_s0(wt) + f.in_off - ch;
                const float2 *in = (const float2 *)f.in;
                // 8-byte cp.async with zero fill: all of a lane's ~18 copies are in flight at once and nothing passes through
                // registers (first version: LDG + STS unrolled by 4, ~5 dependent round trips to L2 per tile -- ncu: the
                // producers spent 55 % of their time there; batches of 10 loads: 2 round trips)
                const uint32_t rs_s = raw_s + (uint32_t)slot * RAWB;
                for (int e = ptid; e < NEL; e += 32 * UC_PROD_WARPS) {
                    const long long j = j0 + f.in_step * e;
                    const bool ok = j >= 0 && j < f.in_limit;
                    cp_async8_zfill(rs_s + 8u * (uint32_t)e, ok ? in + j : in, ok ? 8 : 0);
                }
                cp_async_commit();
                cp_async_wait<0>();
                prod_bar_sync();
            } else if (e_hi - e_lo < NEL) {
                int ch; long long wt;
                split(w, ch, wt);
                const long long s0 = tile_s0(wt);
                const float2 *in = (const float2 *)f.in + (long long)ch * f.in_stride;
                const float2 *hist = (const float2 *)f.hist + (long long)ch * f.hist_stride;
                const int n_plain = e_lo + (NEL - e_hi);
                for (int i = ptid; i < n_plain; i += 32 * UC_PROD_WARPS) {
                    const int e = i < e_lo ? i : e_hi + (i - e_lo);
                    const long long s = s0 + e;
                    float2 v = make_float2(0.0f, 0.0f);
                    if (s >= 0) { if (s < f.n_in) v = __ldg(in + s); }
                    else if (s >= -(long long)f.HL) v = __ldg(hist + (long long)f.HL + s);
                    *reinterpret_cast<float2 *>(rs + 8 * e) = v;
                }
                prod_bar_sync();
            }
            if (e_hi > e_lo) {
                mbar_wait(raw_bar(slot), rph[slot]);
                rph[slot] ^= 1u;
            }
            mbar_wait(empty_bar(stage), ph ^ 1u);
            uint8_t *st_g = gen + (size_t)stage * SB;
            // 8 samples per lane and step: 64 raw bytes -> one 16-byte chunk in each of the 2 NS planes.  A lane's four
            // 16-byte units sit 64 B from its neighbour's: read in lane order they would hit 2 of the 8 bank groups
            // (4-way conflicts, ncu: 64 % of the shared wavefronts were replays).  Lane L therefore starts at unit
            // rot(L) and writes the matching word of each output chunk: loads (8 lanes x 16 B) and stores (32 lanes x 4 B)
            // are both conflict free, and no register has to be re-ordered.
            const int rot = ((lane >> 1) + (lane >> 3)) & 3;
#pragma unroll 2
            for (int c = ptid; c < NEL / 8; c += 32 * UC_PROD_WARPS) {
                const uint8_t *src = rs + 64 * c;
                float re[8], im[8];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 q = *reinterpret_cast<const float4 *>(src + 16 * ((i + rot) & 3));
                    re[2 * i] = q.x; im[2 * i] = q.y; re[2 * i + 1] = q.z; im[2 * i + 1] = q.w;
                }
                const uint32_t off = SmemLayout<64>::swz(16u * (uint32_t)c);
                split_store<NS>(re, st_g, PB, off, rot);
                split_store<NS>(im, st_g + (size_t)NS * PB, PB, off, rot);
            }
            fence_proxy_async();  // plain stores -> visible to the tensor core's (async proxy) operand reads
            mbar_arrive(full_bar(stage));
            prod_bar_sync();      // every producer is done with this raw slot: it may be refilled
            if (!two && ptid == 0) issue_tma(w + wstride, 0);
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            if (two) slot ^= 1;
        }
    } else if (warp == UC_MMA_WARP) {
        // ================= MMA issuer =================
        const uint64_t bdesc0 = smem_desc(tab_s, 128, 256, 0);
        int stage = 0, as = 0;
        uint32_t ph = 0, aph = 0;
        for (long long w = w_begin; w < nwork; w += wstride) {
            mbar_wait(full_bar(stage), ph);
            mbar_wait(acce_bar(as), aph ^ 1u);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t sbase = stage0 + (uint32_t)stage * SB;
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    const uint32_t d0 = tmem + (uint32_t)(as * SETC + part * NCOL);
                    uint64_t ad[NS];
#pragma unroll
                    for (int s = 0; s < NS; ++s) ad[s] = smem_desc(sbase + (uint32_t)((part * NS + s) * PB), 16, 8 * 64, SmemLayout<64>::type);
                    uint64_t bd = bdesc0;
                    // k-step 0 initialises all NCOL columns; everything after accumulates
                    umma_bf16<false>(d0, ad[0], bd, idesc_bf16_f32(128, NCOL));
#pragma unroll
                    for (int s = 1; s < NS; ++s) umma_bf16<true>(d0, ad[s], bd, idesc_bf16_f32(128, 32 * (NS - s)));
                    for (int kk = 1; kk < KS; ++kk) {
                        bd += (NCOL * 32) >> 4;
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            ad[s] += 2;  // 32 bytes = 16 samples along the window
                            umma_bf16<true>(d0, ad[s], bd, idesc_bf16_f32(128, 32 * (NS - s)));
                        }
                    }
                }
                umma_commit(empty_bar(stage));  // the planes may be refilled once these MMAs have read them
                umma_commit(accf_bar(as));      // ... and the accumulator set is complete
            }
            __syncwarp();
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            as ^= 1;
            if (as == 0) aph ^= 1u;
        }
    } else {
        // ================= epilogue: 4 warpgroups; warpgroup wg serves accumulator set wg & 1 and the output columns
        // 16 h .. 16 h + 15 (h = wg >> 1) of every row of that set's tiles =================
        const int ew = warp - UC_EPI_WARP0, wg = ew >> 2, g = wg & 1, h = wg >> 1;
        const int quad = warp & 3;  // TMEM lane quadrant this warp may access
        uint32_t aph = 0;
        long long it = 0;
        for (long long w = w_begin; w < nwork; w += wstride, ++it) {
            if ((it & 1) != g) continue;
            int ch; long long wt;
            split(w, ch, wt);
            float2 *out = (float2 *)f.out + (long long)ch * f.out_stride;
            mbar_wait(accf_bar(g), aph);
            aph ^= 1u;
            tc_fence_after();
            const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(g * SETC + 16 * h);
            const long long m_base = wt * (long long)UC_TILE + (long long)(quad * 32 + (lane >> 2)) * UC_P + 16 * h + 2 * (lane & 3);
            const long long left = f.n_out - m_base;
            const bool full = left > (long long)(24 * UC_P + 10);
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t e[2][NS][8];
#pragma unroll
                for (int part = 0; part < 2; ++part)
#pragma unroll
                    for (int s = 0; s < NS; ++s)
                        tmem_ld_16x256b_x2(tbase + ((uint32_t)(16 * hh) << 16) + (uint32_t)(part * NCOL + 32 * s), e[part][s]);
                tmem_ld_wait();
                if (hh == 1) {
                    // this warp's share of the set is in registers: hand it back to the MMA warp (8 warps arrive)
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acce_bar(g));
                }
#pragma unroll
                for (int cg = 0; cg < 2; ++cg)
#pragma unroll
                    for (int rs = 0; rs < 2; ++rs) {
                        const int i0 = 4 * cg + 2 * rs;
                        const int off = (16 * hh + 8 * rs) * UC_P + 8 * cg;
                        if (full || (long long)off < left) {
                            float y[2][2];
#pragma unroll
                            for (int part = 0; part < 2; ++part)
#pragma unroll
                                for (int q = 0; q < 2; ++q) {
                                    // smallest term first: Sl + Sm, then + Sh
                                    float acc = __uint_as_float(e[part][NS - 1][i0 + q]);
#pragma unroll
                                    for (int s = NS - 2; s >= 0; --s) acc += __uint_as_float(e[part][s][i0 + q]);
                                    y[part][q] = acc;
                                }
                            if (full || (long long)(off + 1) < left) {
                                float4 *dst = reinterpret_cast<float4 *>(out + m_base + off);
                                float4 r = make_float4(y[0][0], y[1][0], y[0][1], y[1][1]);
                                if (f.accumulate) { const float4 o = *dst; r.x += o.x; r.y += o.y; r.z += o.z; r.w += o.w; }
                                *dst = r;
                            } else {
                                float2 r = make_float2(y[0][0], y[1][0]);
                                if (f.accumulate) { const float2 o = out[m_base + off]; r.x += o.x; r.y += o.y; }
                                out[m_base + off] = r;
                            }
                        }
                    }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == UC_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<TMEM_COLS>(tmem);
    }
}

inline uint16_t bf16_rn_bits(float v) {
    uint32_t u;
    std::memcpy(&u, &v, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
inline float bf16_bits_to_float(uint16_t b) {
    const uint32_t u = (uint32_t)b << 16;
    float v;
    std::memcpy(&v, &u, 4);
    return v;
}

}  // namespace

bool fir_umma_c64_applies(int K, int D, bool taps_complex, int ns) {
    if (taps_complex || D != 1 || K < 1 || K > UC_MAX_K || (ns != 2 && ns != 3)) return false;
    int stages, nraw;
    return uc_pick(ns, uc_ksteps(K), &stages, &nraw);
}

// host: [delta 0..1][kk][canonical (32 ns) x 32 B block] of bf16; element (n, kb) of a block sits at
// (n/8)*256 + (kb/8)*128 + (n%8)*16 + (kb%8)*2.  Column n = term * 32 + j: output j of a row, tap term (h, m, l).
bool fir_umma_c64_build_tables(const float *taps, int K, int ns, std::vector<uint8_t> &out) {
    if (!fir_umma_c64_applies(K, 1, false, ns)) return false;
    const int KS = uc_ksteps(K), NCOL = 32 * ns;
    std::vector<uint16_t> term((size_t)ns * K);
    for (int k = 0; k < K; ++k) {
        if (!std::isfinite(taps[k])) return false;
        float r = taps[k];
        for (int s = 0; s < ns; ++s) {
            const uint16_t b = bf16_rn_bits(r);
            term[(size_t)s * K + k] = b;
            r -= bf16_bits_to_float(b);
        }
    }
    out.assign((size_t)2 * KS * NCOL * 32, 0);
    for (int delta = 0; delta < 2; ++delta)
        for (int kk = 0; kk < KS; ++kk) {
            uint8_t *blk = out.data() + ((size_t)delta * KS + kk) * NCOL * 32;
            for (int n = 0; n < NCOL; ++n) {
                const int s = n / 32, j = n % 32;
                for (int kb = 0; kb < 16; ++kb) {
                    const int e = kk * 16 + kb;             // plane element relative to the row start
                    const int t = K - 1 + j + delta - e;    // tap index: element e holds x[row_out0 + e - (K-1) - delta]
                    uint16_t v = 0;
                    if (t >= 0 && t < K) v = term[(size_t)s * K + t];
                    std::memcpy(blk + (n / 8) * 256 + (kb / 8) * 128 + (n % 8) * 16 + (kb % 8) * 2, &v, 2);
                }
            }
        }
    return true;
}

// returns SDR_ERR_UNSUPPORTED when this path does not apply to the call (caller falls back to the CUDA-core kernels)
int fir_umma_c64_launch(const FirArgs &f, int ns, const uint8_t *d_tables, cudaStream_t st, long long branch_tab_stride) {
    if (f.n_out <= 0) return SDR_OK;
    if (f.D != 1 || !fir_umma_c64_applies(f.K, f.D, false, ns)) return SDR_ERR_UNSUPPORTED;
    const bool gather = f.in_step != 0;
    if (((uintptr_t)f.in & 7) || ((uintptr_t)f.out & 15) || (!gather && ((uintptr_t)f.hist & 7)) ||
        (f.n_ch > 1 && ((!gather && (f.in_stride & 1)) || (f.out_stride & 1))))
        return SDR_ERR_UNSUPPORTED;
    const int KS = uc_ksteps(f.K);
    int stages = 2, nraw = 1;
    if (!uc_pick(ns, KS, &stages, &nraw)) return SDR_ERR_UNSUPPORTED;
    const size_t smem = uc_smem_bytes(ns, KS, stages, nraw);
    UcArgs a;
    a.f = f;
    a.KS = KS;
    a.stages = stages;
    a.nraw = nraw;
    a.nel = uc_nel(KS);
    a.plane_bytes = uc_plane_bytes(KS);
    // sample -(K-1) - delta of a tile must sit at a 16-byte aligned address: 8-byte samples, so delta is 0 or 1
    long long d = ((long long)(((uintptr_t)f.in >> 3) & 1) - (long long)(f.K - 1)) % 2;
    if (d < 0) d += 2;
    if (gather) d = 0;  // no bulk copy, no alignment to keep
    a.delta = (int)d;
    a.tab = d_tables + (size_t)d * KS * 32 * ns * 32;
    a.tab_stride = branch_tab_stride;
    a.ntiles = (int)((f.n_out + UC_TILE - 1) / UC_TILE);
    const int sms = current_sm_count();
    const long long nwork = (long long)a.ntiles * f.n_ch;
    if (branch_tab_stride && f.n_ch > sms) return SDR_ERR_UNSUPPORTED;  // every channel needs a CTA of its own
    const unsigned grid = (unsigned)std::min<long long>(nwork, sms);
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kern<<<grid, UC_THREADS, smem, st>>>(a);
        count_launch();
        return launch_status();
    };
    return ns == 2 ? go(fir_umma_c64_kernel<2>) : go(fir_umma_c64_kernel<3>);
}

}  // namespace sdr

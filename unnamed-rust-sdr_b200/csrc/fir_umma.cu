// fir_umma.cu -- K5: fused u8-IQ FIR (+ Decimate) on the 5th-generation tensor cores (tcgen05 / TMEM).
//
// Three kernels: fir_umma_kernel (interleaved bytes; D == 1 and decimation by candidate offsets), fir_umma_poly_kernel
// (decimation on phase planes, D in 5..12) and the opt-in fir_umma_planar_kernel (real taps on I / Q byte planes).
//
// Same reference functions as fir.cu: RtlTcpSignal::next -> signal::Filter::next -> Fir::apply
// (src/rtltcp.rs:158-164, src/signal/adapters/mod.rs:94-96, src/filter/fir.rs:23-32, src/filter/convolve.rs:13-15).
//
// The raw rtl_tcp bytes are NEVER converted: they are the A operand of an integer Toeplitz GEMM.
//
//   y[m] = 2^-(S+7) * sum_k  t[k] * (b[m-k] - 128)          t[k] = round(c[k] * 2^S)  (|t| < 2^23)
//        = 2^-(S+7) * ( sum_k t[k] b[m-k]  -  128 sum_k t[k] )
//
//   * A (M = 128 rows, K-major, u8): row i of a tile is the window of interleaved I,Q BYTES that starts 2P bytes after
//     row i-1.  A shared-memory matrix descriptor whose rows overlap (row pitch 2P bytes inside ONE flat copy of the
//     input: pitch 16 B = no swizzle, 32 B = SWIZZLE_32B, 64 B = SWIZZLE_64B) reads exactly that Hankel matrix, so the
//     input is staged once, untouched, by cp.async straight from global memory (scripts/probes/umma_toeplitz_probe.cu
//     is the hardware check: the swizzle XOR is a function of the absolute shared address, so overlapping rows agree).
//   * B (N = 6P columns, K-major, s8): banded Toeplitz block of the integer taps, split into three balanced base-256
//     digits; column (digit d, phase j, part q) holds digit d of the taps that produce the I (q=0) or Q (q=1) part of
//     output P*i + j.  Real taps touch only the I (or Q) bytes of the window; complex taps touch both
//     (y.re = x.re c.re - x.im c.im, y.im = x.re c.im + x.im c.re: the signs live in the table).
//   * D (TMEM, s32): exact integer sums.  |sum| <= 255*128*K < 2^31 and |sum - 128 sum_k d| <= 2^14 K < 2^23 for
//     K <= 511, so the epilogue combines digits 0 and 1 in s32, converts (one I2F, and the 1.5*2^23 magic-number add for
//     digit 2) and joins them with one FFMA: the result is the exactly-accumulated dot product rounded ~once -- closer
//     to the f64 truth than the reference's own sequential f32 sum (tests/test_gpu_fir.py bars: 1e-5 relative, and
//     <= 4x the reference's error), and independent of how the stream is cut into calls.
//
// Decimation (signal::Decimate fused behind the filter, src/signal/adapters/mod.rs:30-37): rows stay R = 32 samples
// apart (a matrix descriptor cannot step by D), and the B columns are the CANDIDATE offsets inside a row at which a
// kept output can fall: kept output m sits D*m samples after output 0, i.e. in row (D m) div R at offset (D m) mod R, a
// multiple of g = gcd(D, R).  Only those R/g offsets get columns (D = 10: 16 of 32, N = 96); the epilogue keeps a
// candidate iff its offset from output 0 is a multiple of D (multiply-shift modulo) and stores it at out[offset / D].
//
// Warp roles (one persistent CTA per SM, 640 threads):
//   warps 0..2  producers: cp.async 16-byte chunks global -> (swizzled) stage, completion on an mbarrier
//                          (cp.async.mbarrier.arrive.noinc); history / zero padding at the stream start by plain stores
//   warp 3      MMA issuer: one elected lane (elect.sync) issues KS * MB tcgen05.mma.kind::i8 per tile with running
//                          descriptors; tcgen05.commit frees the stage and publishes the accumulator set
//   warps 4..19 four epilogue warpgroups (two accumulator sets x two halves of a tile): tcgen05.ld.16x256b fragments ->
//               digits -> f32 -> global stores straight from registers (4 threads = one 32-byte sector)
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "kernels.h"
#include "ptx.cuh"

namespace sdr {

namespace {

constexpr int UM_STAGES = 4;            // at most; fewer when the tap tables leave less shared memory
constexpr int UM_ACC_COLS = 192;       // TMEM columns per accumulator set = MB * 6 PC
constexpr int UM_PROD_WARPS = 3;                   // producer warps (one was LDGSTS-issue bound: 8-10 B/cycle/SM)
constexpr int UM_MMA_WARP = UM_PROD_WARPS;         // the MMA-issuing warp
constexpr int UM_EPI_WARP0 = UM_PROD_WARPS + 1;    // 16 epilogue warps follow
constexpr int UM_THREADS = (UM_PROD_WARPS + 1 + 16) * 32;
constexpr int UM_MAX_K = 511;

struct UmArgs {
    FirArgs f;
    const uint8_t *tab;  // this call's alignment variant: KS blocks of N*32 bytes in canonical no-swizzle K-major order
    int KS;              // k-steps of 32 bytes = 16 samples
    int delta;           // window start is `delta` samples left of the first needed sample (16-byte alignment)
    int ntiles;          // tiles per channel
    int stage_bytes;     // one stage: the tile's window starts + (KS*32 B) halo, multiple of 1024 (swizzle period)
    long long n_rows;    // window rows per channel that hold at least one kept output
    int stages;          // input stages in the ring (2..UM_STAGES)
    unsigned dmagic;     // floor(2^32 / D) + 1: n / D == umulhi(n, dmagic) for n < 2^17, D <= 4096
    int magic[2][3];     // [part]: {-(256 C1 + C0), unused, 0x4B400000 - C2}, C_d = 128 * sum of that column's digit-d taps
    float sc[3];         // 2^-(S+7) * {1, 256, 65536}
    // TMA (fir_umma_kernel): interior tiles are staged by tma_nbox tensor copies of tma_rows window rows each
    int use_tma = 0, tma_rows = 0, tma_nbox = 0;
    int tma_shift = 0;   // bytes the tensor map's base sits below the caller's `in` (16-byte alignment of the map)
    int tma_need = 0;    // window rows a tile really reads (the boxes are rounded up to multiples of 8 rows)
    long long tma_rows_total = 0;  // rows of the map: a tile whose needed rows reach beyond it is staged by cp.async
};

// one stage holds the 128*MB window starts of a tile, R samples apart, plus the KS*32-byte halo of the last row
__host__ __device__ constexpr int um_stage_bytes(int R, int PC, int KS) {
    return (2 * R * (128 * (32 / PC) - 1) + 32 * KS + 1023) / 1024 * 1024;
}
__host__ __device__ constexpr size_t um_smem_bytes(int R, int PC, int KS, bool dec, int stages = UM_STAGES) {
    // tables + stages + 1 KB alignment slack + barriers (the epilogue stores straight from registers)
    (void)dec;
    return (size_t)KS * 6 * PC * 32 + (size_t)stages * um_stage_bytes(R, PC, KS) + 1024 + 256;
}

// R = samples between window rows (8 / 16 / 32: no / 32-byte / 64-byte swizzle), PC = output candidates per row
// (PC == R when D == 1), DEC = decimating epilogue.
// work item w = ch * ntiles + tile.  The single-channel case (the u8 stream configs) skips the 64-bit division, which
// is ~100 instructions on the per-tile path of every role.
__device__ __forceinline__ void split_work(long long w, int ntiles, int n_ch, int &ch, long long &tile) {
    if (n_ch == 1) { ch = 0; tile = w; }
    else if (w <= 0x7fffffffLL) { const unsigned c = (unsigned)w / (unsigned)ntiles; ch = (int)c; tile = (long long)((unsigned)w - c * (unsigned)ntiles); }
    else { ch = (int)(w / ntiles); tile = w - (long long)ch * ntiles; }
}

template <int R, int PC, bool DEC>
__global__ void __launch_bounds__(UM_THREADS, 1) fir_umma_kernel(const UmArgs a, const __grid_constant__ CUtensorMap tmap) {
    constexpr int P = R;                     // (name kept from the D == 1 derivation: outputs per row when PC == R)
    constexpr int MB = 32 / PC;              // 128-row blocks per tile
    constexpr int N = 6 * PC;                // MMA N: 3 digits x PC candidates x (I, Q)
    constexpr int ROWB = 2 * R;              // bytes between window rows
    constexpr int TILE_ROWS = 128 * MB;
    const int SB = a.stage_bytes, NST = a.stages;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * UM_STAGES + 4];
    __shared__ uint32_t tmem_base_s;
    const FirArgs &f = a.f;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KS = a.KS;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;  // stages first: 1024-aligned for the swizzle modes
    const uint32_t stage0 = base;
    const uint32_t tab_s = stage0 + NST * SB;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));        // generic pointer to `base`
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (UM_STAGES + s); };
    auto accf_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + s); };
    auto acce_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + 2 + s); };

    // ---- one-time setup ----
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.tab);
        uint4 *dst = reinterpret_cast<uint4 *>(gen + NST * SB);
        for (int i = tid; i < KS * N * 2; i += UM_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < UM_STAGES; ++s) { mbar_init(full_bar(s), 32 * UM_PROD_WARPS); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(accf_bar(s), 1); mbar_init(acce_bar(s), 8); }
        mbar_init_fence();
    }
    if (warp == UM_MMA_WARP) {
        tmem_alloc<512>(smem_u32(&tmem_base_s));
    }
    fence_proxy_async();  // the tap tables were written through the generic proxy, tcgen05.mma reads through the async one
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    const long long nwork = (long long)a.ntiles * f.n_ch;
    const long long wstride = gridDim.x;

    if (warp < UM_PROD_WARPS) {
        // ================= producers =================
        const int ptid = warp * 32 + lane;
        const int nchunks = (ROWB * (128 * MB - 1) + 32 * KS + 15) / 16;
        int stage = 0;
        uint32_t ph = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride) {
            int ch; long long wt;
            split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
            const long long w0 = f.first - (f.K - 1) - a.delta + wt * (long long)(TILE_ROWS * R);  // multiple of 8
            const unsigned char *in = (const unsigned char *)f.in + (long long)ch * f.in_stride * 2;
            const unsigned char *hist = (const unsigned char *)f.hist + (long long)ch * f.hist_stride * 2;
            mbar_wait(empty_bar(stage), ph ^ 1u);
            const uint32_t sbase = stage0 + (uint32_t)stage * SB;
            bool slow = false;
            if (w0 >= 0 && w0 + 8LL * nchunks <= f.n_in && a.use_tma &&
                (2 * w0 + a.tma_shift) / ROWB + a.tma_need <= a.tma_rows_total) {
                // interior tile, TMA: the sliding window with its tap-length halo is ONE tensor copy (two when it has
                // more than 256 rows) issued by one thread.  The map views the byte stream as rows of ROWB bytes that
                // may start at any 16-byte offset ({ROWB, ROWB/16 sub-offsets, rows[, channel]}), the box is
                // {ROWB, 1, rows}, and the map's swizzle mode is the A descriptor's: the bytes land exactly where the
                // cp.async loop below puts them.  Rows past the end of the stream are zero-filled by the hardware
                // (they feed only outputs that are never stored).
                if (ptid == 0) {
                    const long long b0 = 2 * w0 + a.tma_shift;  // byte offset from the map's base: a multiple of 16
                    const int c1 = (int)((b0 / 16) % (ROWB / 16)), c2 = (int)(b0 / ROWB);
                    mbar_arrive_expect_tx(full_bar(stage), (uint32_t)(a.tma_nbox * a.tma_rows * ROWB));
                    for (int i = 0; i < a.tma_nbox; ++i) {
                        const uint32_t dst = sbase + (uint32_t)(i * a.tma_rows * ROWB);
                        if (f.n_ch == 1) tma_load_3d(dst, &tmap, 0, c1, c2 + i * a.tma_rows, full_bar(stage));
                        else tma_load_4d(dst, &tmap, 0, c1, c2 + i * a.tma_rows, ch, full_bar(stage));
                    }
                } else {
                    mbar_arrive(full_bar(stage));
                }
                if (++stage == NST) { stage = 0; ph ^= 1u; }
                continue;
            } else if (w0 >= 0 && w0 + 8LL * nchunks <= f.n_in) {
                // interior tile (all but the first / last of a block): nothing but address arithmetic and LDGSTS
                const unsigned char *src = in + 2 * w0;
#pragma unroll 4
                for (int c = ptid; c < nchunks; c += 32 * UM_PROD_WARPS)
                    cp_async16_s(sbase + SmemLayout<ROWB>::swz(16u * (uint32_t)c), src + 16 * c);
            } else {
                for (int c = ptid; c < nchunks; c += 32 * UM_PROD_WARPS) {
                    const long long s0 = w0 + 8LL * c;
                    const uint32_t off = SmemLayout<ROWB>::swz(16u * (uint32_t)c);
                    if (s0 >= 0 && s0 + 8 <= f.n_in) {
                        cp_async16_s(sbase + off, in + 2 * s0);
                    } else if (s0 < f.n_in) {
                        // stream start (carried history, then "zero" samples = byte pair 128,128) or the ragged end
                        unsigned short h[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const long long s = s0 + i;
                            unsigned short v = 0x8080;
                            if (s >= 0) { if (s < f.n_in) v = *reinterpret_cast<const unsigned short *>(in + 2 * s); }
                            else if (s >= -(long long)f.HL) v = *reinterpret_cast<const unsigned short *>(hist + 2 * ((long long)f.HL + s));
                            h[i] = v;
                        }
                        uint4 q;
                        q.x = h[0] | ((unsigned)h[1] << 16); q.y = h[2] | ((unsigned)h[3] << 16);
                        q.z = h[4] | ((unsigned)h[5] << 16); q.w = h[6] | ((unsigned)h[7] << 16);
                        *reinterpret_cast<uint4 *>(gen + (size_t)stage * SB + off) = q;
                        slow = true;
                    }
                    // chunks entirely past the end feed only rows whose outputs are never stored: left as they are
                }
            }
            if (slow) fence_proxy_async();
            cp_async_arrive_noinc(full_bar(stage));
            if (++stage == NST) { stage = 0; ph ^= 1u; }
        }
        cp_async_wait_all();
    } else if (warp == UM_MMA_WARP) {
        // ================= MMA issuer =================
        const uint32_t idesc = idesc_u8s8_s32(128, N);
        const uint64_t bdesc0 = smem_desc(tab_s, 128, 256, 0);
        int stage = 0, as = 0;
        uint32_t ph = 0, aph = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride) {
            mbar_wait(full_bar(stage), ph);
            mbar_wait(acce_bar(as), aph ^ 1u);
            tc_fence_after();
            if (elect_one()) {
                // running descriptors: the issuing thread's uniform-datapath work per MMA is two 64-bit adds of
                // constants (recomputing them from kk cost ~130 cycles per MMA: the real limit of MMA-heavy tiles)
                uint64_t ad = smem_desc(stage0 + (uint32_t)stage * SB, 16, 8 * ROWB, SmemLayout<ROWB>::type);
                uint64_t bd = bdesc0;
                const uint32_t d0 = tmem + (uint32_t)(as * UM_ACC_COLS);
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) umma_i8<false>(d0 + mb * N, ad + (uint64_t)((mb * 128 * ROWB) >> 4), bd, idesc);
                for (int kk = 1; kk < KS; ++kk) {
                    ad += 2;               // 32 bytes along the window
                    bd += (N * 32) >> 4;   // next tap block
#pragma unroll
                    for (int mb = 0; mb < MB; ++mb) umma_i8<true>(d0 + mb * N, ad + (uint64_t)((mb * 128 * ROWB) >> 4), bd, idesc);
                }
                umma_commit(empty_bar(stage));  // the stage may be refilled once these MMAs have read it
                umma_commit(accf_bar(as));      // ... and the accumulator set is complete
            }
            __syncwarp();
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            as ^= 1;
            if (as == 0) aph ^= 1u;
        }
    } else {
        // ================= epilogue: 4 warpgroups; warpgroup wg works on accumulator set wg & 1 and converts the
        // pieces 2h, 2h+1 (h = wg >> 1) of every tile of that set.  A piece = 8 candidates (16 columns of each digit) of
        // one 128-row block; a tile has 4 (MB * PC/8).  Both halves of a set run concurrently: twice the warps hide the
        // TMEM / shared / conversion latencies, and the set returns to the MMA warp in half the time. =================
        const int ew = warp - UM_EPI_WARP0, wg = ew >> 2, g = wg & 1, h = wg >> 1;
        const int quad = warp & 3;  // TMEM lane quadrant this warp may access
        constexpr int PPB = PC / 8;                  // pieces per 128-row block
        const float sc0 = a.sc[0], sc2 = a.sc[2];
        const int c10[2] = {a.magic[0][0], a.magic[1][0]}, m2[2] = {a.magic[0][2], a.magic[1][2]};
        uint32_t aph = 0;
        long long it = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride, ++it) {
            if ((it & 1) != g) continue;
            int ch; long long wt;
            split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
            const long long row0 = wt * (long long)TILE_ROWS;  // first window row of the tile
            float2 *out = (float2 *)f.out + (long long)ch * f.out_stride;
            mbar_wait(accf_bar(g), aph);
            aph ^= 1u;
            tc_fence_after();
            const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(g * UM_ACC_COLS);
            // DEC: kept output m sits at sample offset D*m from output 0; the tile starts at offset row0*R
            unsigned rem0 = 0;
            long long mt0 = 0;
            if constexpr (DEC) {
                const long long tp = row0 * (long long)R;
                mt0 = tp / f.D;
                rem0 = (unsigned)(tp - mt0 * f.D);
            }
#pragma unroll
            for (int pj = 0; pj < 2; ++pj) {
                const int pi = 2 * h + pj, mb = pi / PPB, pc = pi % PPB;
                // No shared-memory staging: the 16x256b fragment shape hands every thread whole (I, Q) column pairs of
                // two rows; 4 neighbouring threads hold 4 consecutive candidates of one row.  D == 1: 32 contiguous
                // output bytes (one full sector) per 4 threads, 8 sectors per store instruction.  The shared-memory
                // port is left to the MMA operand fetch and the producers.
                uint32_t e[2][3][8];
                const uint32_t col = tbase + (uint32_t)(mb * N + 16 * pc);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                    for (int dg = 0; dg < 3; ++dg) tmem_ld_16x256b_x2(col + ((uint32_t)(16 * hh) << 16) + dg * 2 * PC, e[hh][dg]);
                tmem_ld_wait();
                if (pj == 1) {
                    // this warp's share of the set is in registers: hand it back to the MMA warp (8 warps arrive)
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acce_bar(g));
                }
                if constexpr (!DEC) {
                    // D == 1: output index = (row0 + row) * P + u.  Everything but (16 hh + 8 rs) * P + 4 cg is folded
                    // into one per-thread pointer per piece, so a store is STG [base + immediate]; a tile that lies
                    // entirely inside the call (all but the last) needs no per-output bound test either.  (Computing
                    // index, address and bound per output cost as many instructions as the conversion itself in this
                    // epilogue-bound kernel.)
                    const long long m_base = row0 * (long long)P + (long long)(mb * 128 + quad * 32 + (lane >> 2)) * P +
                                             8 * pc + (lane & 3);
                    float2 *ob = out + m_base;
                    const long long left = f.n_out - m_base;  // outputs from this thread's first one to the end
                    const bool full = left > (long long)(24 * P + 4);
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                        for (int cg = 0; cg < 2; ++cg)
#pragma unroll
                            for (int rs = 0; rs < 2; ++rs) {
                                const int i0 = 4 * cg + 2 * rs;
                                const int off = (16 * hh + 8 * rs) * P + 4 * cg;
                                if (full || (long long)off < left) {
                                    const float fI = (float)((int)(e[hh][1][i0] << 8) + (int)e[hh][0][i0] + c10[0]);
                                    const float fQ = (float)((int)(e[hh][1][i0 + 1] << 8) + (int)e[hh][0][i0 + 1] + c10[1]);
                                    const float gI = __int_as_float((int)e[hh][2][i0] + m2[0]) - 12582912.0f;
                                    const float gQ = __int_as_float((int)e[hh][2][i0 + 1] + m2[1]) - 12582912.0f;
                                    ob[off] = make_float2(fmaf(gI, sc2, fI * sc0), fmaf(gQ, sc2, fQ * sc0));
                                }
                            }
                } else
#pragma unroll
                for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                    for (int cg = 0; cg < 2; ++cg)
#pragma unroll
                        for (int rs = 0; rs < 2; ++rs) {
                            const int i0 = 4 * cg + 2 * rs;
                            const int row = mb * 128 + quad * 32 + 16 * hh + 8 * rs + (lane >> 2);  // row inside the tile
                            const int u = 8 * pc + 4 * cg + (lane & 3);                              // candidate
                            long long m;
                            bool keep;
                            if constexpr (DEC) {
                                // offset of this candidate from output 0, modulo D by multiply-shift (n < 2^17, D <= 4096)
                                const unsigned n = rem0 + (unsigned)(row * R + (R / PC) * u);
                                const unsigned q = __umulhi(n, a.dmagic);
                                m = mt0 + q;
                                keep = (n - q * (unsigned)f.D == 0u) && m < f.n_out;
                            } else {
                                m = (row0 + row) * (long long)P + u;
                                keep = m < f.n_out;
                            }
                            if (keep) {
                                // digits 0 and 1 combine exactly in s32 ((A1 << 8) + A0, |.| < 2^31 for K <= 511; wrap-around
                                // safe); digit 2 (|A2| < 2^23) converts with the 1.5 * 2^23 magic add: one I2F per value
                                const float fI = (float)((int)(e[hh][1][i0] << 8) + (int)e[hh][0][i0] + c10[0]);
                                const float fQ = (float)((int)(e[hh][1][i0 + 1] << 8) + (int)e[hh][0][i0 + 1] + c10[1]);
                                const float gI = __int_as_float((int)e[hh][2][i0] + m2[0]) - 12582912.0f;
                                const float gQ = __int_as_float((int)e[hh][2][i0 + 1] + m2[1]) - 12582912.0f;
                                out[m] = make_float2(fmaf(gI, sc2, fI * sc0), fmaf(gQ, sc2, fQ * sc0));
                            }
                        }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == UM_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

// =====================================================================================================================
// Planar variant for REAL taps (opt-in: SDR_FIR_PLANAR).  With interleaved I,Q bytes half of every real-tap B column
// is zero (an I output never touches a Q byte): half of the tensor work and of the tap-table operand traffic is wasted.
// Here the producers split each 16-byte chunk into its 8 I and 8 Q bytes (two PRMT pairs) and keep two byte planes per
// stage; a k-step is 32 SAMPLES of one plane, both planes multiply the same B block (N = 3 PC) into their own
// accumulator columns.  Rows are R BYTES apart inside a plane (16 / 32 / 64: no swizzle / SWIZZLE_32B / SWIZZLE_64B),
// so a row spans twice the samples of the interleaved kernel: for 255 taps the MMA count per sample halves and the
// tables shrink 4x.  Everything downstream of the MMAs (hand-over, conversion, staging, stores) is the interleaved
// kernel's, and the results are bit-identical (test_planar_and_interleaved_...).
// MEASURED (round 1): not faster.  ncu (profiles/r01_prof_fir_planar_k255.txt): tensor pipe 32 %, epilogue warps 62 %
// waiting for accumulators, producers stalled on LDS -> PRMT.  The limit of this kernel family at 255 taps is the
// 128 B/cycle shared-memory port that MMA operand fetch (140-190 KB per 4096-sample tile), the epilogue staging (64 KB)
// and the producers share; the raw-ring -> plane conversion adds 17 KB per tile to it and puts an LDS on the
// producers' critical path.  C1 392 vs 490, C3 483 vs 588, 255 taps D=1 343 vs 321-377 Gsamples/s: it stays opt-in.
// =====================================================================================================================
// one plane of a stage: the 128*MB window starts R bytes apart + the KS*32-byte halo, 1024-aligned
__host__ __device__ constexpr int um_plane_bytes(int R, int PC, int KS) {
    return (R * (128 * (32 / PC) - 1) + 32 * KS + 1023) / 1024 * 1024;
}
// raw ring slot: the tile's interleaved bytes as they arrive from HBM (cp.async), before the split into planes
__host__ __device__ constexpr int um_raw_bytes(int R, int PC, int KS) {
    return (R * (128 * (32 / PC) - 1) + 32 * KS + 7) / 8 * 16;
}
constexpr int UM_RAW_SLOTS = 3;
__host__ __device__ constexpr size_t um_planar_smem_bytes(int R, int PC, int KS, bool dec, int stages) {
    return (size_t)KS * 3 * PC * 32 + (size_t)stages * 2 * um_plane_bytes(R, PC, KS) +
           (dec ? (size_t)16 * 6144 : (size_t)16 * 32 * 8 * 16) + (size_t)UM_RAW_SLOTS * um_raw_bytes(R, PC, KS) + 1024 + 256;
}

template <int R, int PC, bool DEC>
__global__ void __launch_bounds__(UM_THREADS, 1) fir_umma_planar_kernel(const UmArgs a) {
    constexpr int P = R;                     // D == 1: outputs per row
    constexpr int MB = 32 / PC;              // 128-row blocks per tile
    constexpr int N = 3 * PC;                // MMA N per plane: 3 digits x PC candidates
    constexpr int TILE_ROWS = 128 * MB;
    const int SB = a.stage_bytes, NST = a.stages, PB = SB / 2;  // stage = I plane, Q plane
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * UM_STAGES + 4];
    __shared__ uint32_t tmem_base_s;
    const FirArgs &f = a.f;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KS = a.KS;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stage0 = base;
    const uint32_t tab_s = stage0 + NST * SB;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (UM_STAGES + s); };
    auto accf_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + s); };
    auto acce_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + 2 + s); };

    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.tab);
        uint4 *dst = reinterpret_cast<uint4 *>(gen + NST * SB);
        for (int i = tid; i < KS * N * 2; i += UM_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < UM_STAGES; ++s) { mbar_init(full_bar(s), 32 * UM_PROD_WARPS); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(accf_bar(s), 1); mbar_init(acce_bar(s), 8); }
        mbar_init_fence();
    }
    if (warp == UM_MMA_WARP) {
        tmem_alloc<512>(smem_u32(&tmem_base_s));
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const long long nwork = (long long)a.ntiles * f.n_ch;
    const long long wstride = gridDim.x;

    if (warp < UM_PROD_WARPS) {
        // ================= producers =================
        // Every lane owns the chunks c = ptid + 96 i of each tile, end to end: cp.async them (two tiles ahead) into a
        // raw ring slot, wait for its OWN copies (cp.async.wait_group), split each 16-byte chunk into 8 I + 8 Q bytes
        // and store them into the stage's planes.  No producer-to-producer synchronisation, deep asynchronous loads.
        const int ptid = warp * 32 + lane;
        const int nchunks = (R * (TILE_ROWS - 1) + 32 * KS + 7) / 8;  // 8-sample chunks a tile touches
        const int RAWB = 16 * nchunks;
        uint8_t *raw0 = gen + (size_t)NST * SB + (size_t)KS * N * 32 + (size_t)16 * (DEC ? 6144 : 32 * 8 * 16);
        auto issue = [&](long long w, int slot) {
            if (w < nwork) {
                int ch; long long wt;
                split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
                const long long w0 = f.first - (f.K - 1) - a.delta + wt * (long long)(TILE_ROWS * R);  // multiple of 8
                const unsigned char *in = (const unsigned char *)f.in + (long long)ch * f.in_stride * 2;
                const unsigned char *hist = (const unsigned char *)f.hist + (long long)ch * f.hist_stride * 2;
                uint8_t *rs = raw0 + (size_t)slot * RAWB;
                const uint32_t rs_s = smem_u32(rs);
                if (w0 >= 0 && w0 + 8LL * nchunks <= f.n_in) {
                    const unsigned char *src = in + 2 * w0;
#pragma unroll 4
                    for (int c = ptid; c < nchunks; c += 32 * UM_PROD_WARPS) cp_async16_s(rs_s + 16u * c, src + 16 * c);
                } else {
                    for (int c = ptid; c < nchunks; c += 32 * UM_PROD_WARPS) {
                        const long long s0 = w0 + 8LL * c;
                        if (s0 >= 0 && s0 + 8 <= f.n_in) {
                            cp_async16_s(rs_s + 16u * c, in + 2 * s0);
                        } else if (s0 < f.n_in) {
                            // stream start (carried history, then "zero" samples = byte pair 128,128) or the ragged end
                            unsigned short h[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const long long s = s0 + i;
                                unsigned short v = 0x8080;
                                if (s >= 0) { if (s < f.n_in) v = *reinterpret_cast<const unsigned short *>(in + 2 * s); }
                                else if (s >= -(long long)f.HL) v = *reinterpret_cast<const unsigned short *>(hist + 2 * ((long long)f.HL + s));
                                h[i] = v;
                            }
                            uint4 q;
                            q.x = h[0] | ((unsigned)h[1] << 16); q.y = h[2] | ((unsigned)h[3] << 16);
                            q.z = h[4] | ((unsigned)h[5] << 16); q.w = h[6] | ((unsigned)h[7] << 16);
                            *reinterpret_cast<uint4 *>(rs + 16 * c) = q;  // read back by this same lane
                        }
                        // chunks entirely past the end feed only rows whose outputs are never stored: left as they are
                    }
                }
            }
            cp_async_commit();
        };
        issue(blockIdx.x, 0);
        issue(blockIdx.x + wstride, 1);
        int stage = 0, slot = 0;
        uint32_t ph = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride) {
            int s2 = slot + 2;
            if (s2 >= UM_RAW_SLOTS) s2 -= UM_RAW_SLOTS;
            issue(w + 2 * wstride, s2);
            cp_async_wait<2>();  // this lane's chunks of tile w have landed
            mbar_wait(empty_bar(stage), ph ^ 1u);
            uint8_t *pI = gen + (size_t)stage * SB, *pQ = pI + PB;
            const uint8_t *rs = raw0 + (size_t)slot * RAWB;
#pragma unroll 2
            for (int c = ptid; c < nchunks; c += 32 * UM_PROD_WARPS) {
                const uint4 q = *reinterpret_cast<const uint4 *>(rs + 16 * c);  // words = I0 Q0 I1 Q1
                const uint32_t i_lo = __byte_perm(q.x, q.y, 0x6420), i_hi = __byte_perm(q.z, q.w, 0x6420);
                const uint32_t q_lo = __byte_perm(q.x, q.y, 0x7531), q_hi = __byte_perm(q.z, q.w, 0x7531);
                const uint32_t off = SmemLayout<R>::swz((8u * (uint32_t)c) & ~15u) | ((8u * (uint32_t)c) & 8u);
                *reinterpret_cast<uint2 *>(pI + off) = make_uint2(i_lo, i_hi);
                *reinterpret_cast<uint2 *>(pQ + off) = make_uint2(q_lo, q_hi);
            }
            fence_proxy_async();  // plain stores -> visible to the tensor core's (async proxy) operand reads
            mbar_arrive(full_bar(stage));
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            if (++slot == UM_RAW_SLOTS) slot = 0;
        }
        cp_async_wait_all();
    } else if (warp == UM_MMA_WARP) {
        // ================= MMA issuer =================
        const uint32_t idesc = idesc_u8s8_s32(128, N);
        const uint64_t bdesc0 = smem_desc(tab_s, 128, 256, 0);
        int stage = 0, as = 0;
        uint32_t ph = 0, aph = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride) {
            mbar_wait(full_bar(stage), ph);
            mbar_wait(acce_bar(as), aph ^ 1u);
            tc_fence_after();
            if (elect_one()) {
                uint64_t aI = smem_desc(stage0 + (uint32_t)stage * SB, 16, 8 * R, SmemLayout<R>::type);
                uint64_t aQ = smem_desc(stage0 + (uint32_t)stage * SB + PB, 16, 8 * R, SmemLayout<R>::type);
                uint64_t bd = bdesc0;
                const uint32_t d0 = tmem + (uint32_t)(as * UM_ACC_COLS);
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) {
                    umma_i8<false>(d0 + mb * 2 * N, aI + (uint64_t)((mb * 128 * R) >> 4), bd, idesc);
                    umma_i8<false>(d0 + mb * 2 * N + N, aQ + (uint64_t)((mb * 128 * R) >> 4), bd, idesc);
                }
                for (int kk = 1; kk < KS; ++kk) {
                    aI += 2; aQ += 2;
                    bd += (N * 32) >> 4;
#pragma unroll
                    for (int mb = 0; mb < MB; ++mb) {
                        umma_i8<true>(d0 + mb * 2 * N, aI + (uint64_t)((mb * 128 * R) >> 4), bd, idesc);
                        umma_i8<true>(d0 + mb * 2 * N + N, aQ + (uint64_t)((mb * 128 * R) >> 4), bd, idesc);
                    }
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
        // ================= epilogue (see fir_umma_kernel) =================
        const int ew = warp - UM_EPI_WARP0, wg = ew >> 2, g = wg & 1, h = wg >> 1;
        const int quad = warp & 3;
        constexpr int PPB = PC / 8;
        constexpr int SW = 8;  // P >= 16 always here
        constexpr int STG_BYTES = DEC ? 6144 : 32 * SW * 16;
        uint8_t *stg = gen + (size_t)NST * SB + (size_t)KS * N * 32 + (size_t)ew * STG_BYTES;
        const float sc0 = a.sc[0], sc2 = a.sc[2];
        const int c10 = a.magic[0][0], m2 = a.magic[0][2];
        uint32_t aph = 0;
        long long it = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride, ++it) {
            if ((it & 1) != g) continue;
            int ch; long long wt;
            split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
            const long long row0 = wt * (long long)TILE_ROWS;
            float2 *out = (float2 *)f.out + (long long)ch * f.out_stride;
            mbar_wait(accf_bar(g), aph);
            aph ^= 1u;
            tc_fence_after();
            const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(g * UM_ACC_COLS);
            long long pos0 = 0, m_lo = 0;
            int n_m = 0;
#pragma unroll
            for (int pj = 0; pj < 2; ++pj) {
                const int pi = 2 * h + pj, mb = pi / PPB, pc = pi % PPB;
                uint32_t dI[3][8], dQ[3][8];
                {
                    const uint32_t col = tbase + (uint32_t)(mb * 2 * N + 8 * pc);
#pragma unroll
                    for (int dg = 0; dg < 3; ++dg) {
                        tmem_ld_32x32b_x8(col + dg * PC, dI[dg]);
                        tmem_ld_32x32b_x8(col + N + dg * PC, dQ[dg]);
                    }
                    tmem_ld_wait();
                }
                if (pj == 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acce_bar(g));
                }
                if constexpr (DEC) {
                    constexpr int G = R / PC, LG = (G == 1) ? 0 : (G == 2) ? 1 : 2;
                    uint4 *srow = reinterpret_cast<uint4 *>(stg) + lane * 12;
#pragma unroll
                    for (int dg = 0; dg < 3; ++dg)
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            int c = dg * 4 + q + (lane % 12);
                            if (c >= 12) c -= 12;
                            srow[c] = make_uint4(dI[dg][2 * q], dQ[dg][2 * q], dI[dg][2 * q + 1], dQ[dg][2 * q + 1]);
                        }
                    __syncwarp();
                    if (pj == 0 || PPB == 1) {
                        pos0 = (row0 + mb * 128 + quad * 32) * (long long)R;
                        m_lo = (pos0 + f.D - 1) / f.D;
                        n_m = (int)((pos0 + 32 * R + f.D - 1) / f.D - m_lo);
                    }
                    for (int i = lane; i < n_m; i += 32) {
                        const long long m = m_lo + i;
                        const int pos = (int)(m * f.D - pos0);
                        const int r = pos / R, u = (pos % R) >> LG;
                        if ((u >> 3) == pc && m < f.n_out) {
                            const int uu = u & 7, cb = uu >> 1, rot = r % 12;
                            const unsigned char *rowp = stg + r * 192 + (uu & 1) * 8;
                            int c0 = cb + rot, c1 = 4 + cb + rot, c2 = 8 + cb + rot;
                            if (c0 >= 12) c0 -= 12;
                            if (c1 >= 12) c1 -= 12;
                            if (c2 >= 12) c2 -= 12;
                            const uint2 a0 = *reinterpret_cast<const uint2 *>(rowp + c0 * 16);
                            const uint2 a1 = *reinterpret_cast<const uint2 *>(rowp + c1 * 16);
                            const uint2 a2 = *reinterpret_cast<const uint2 *>(rowp + c2 * 16);
                            const float fI = (float)((int)(a1.x << 8) + (int)a0.x + c10);
                            const float fQ = (float)((int)(a1.y << 8) + (int)a0.y + c10);
                            const float gI = __int_as_float((int)a2.x + m2) - 12582912.0f;
                            const float gQ = __int_as_float((int)a2.y + m2) - 12582912.0f;
                            out[m] = make_float2(fmaf(gI, sc2, fI * sc0), fmaf(gQ, sc2, fQ * sc0));
                        }
                    }
                    __syncwarp();
                } else {
                    float y[16];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const float fI = (float)((int)(dI[1][u] << 8) + (int)dI[0][u] + c10);
                        const float fQ = (float)((int)(dQ[1][u] << 8) + (int)dQ[0][u] + c10);
                        const float gI = __int_as_float((int)dI[2][u] + m2) - 12582912.0f;
                        const float gQ = __int_as_float((int)dQ[2][u] + m2) - 12582912.0f;
                        y[2 * u] = fmaf(gI, sc2, fI * sc0);
                        y[2 * u + 1] = fmaf(gQ, sc2, fQ * sc0);
                    }
                    const int cl0 = 4 * (pc % (SW / 4));
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int c = cl0 + q;
                        *reinterpret_cast<float4 *>(stg + ((size_t)lane * SW + (c ^ (lane & 7))) * 16) =
                            make_float4(y[4 * q], y[4 * q + 1], y[4 * q + 2], y[4 * q + 3]);
                    }
                    if (cl0 + 4 == SW) {
                        __syncwarp();
                        const int phase0 = (P == 32) ? 16 * h : 0;
                        const long long mrow = (row0 + mb * 128 + quad * 32) * (long long)P;
                        float4 val[SW];
#pragma unroll
                        for (int i = 0; i < SW; ++i) {
                            const int q = i * 32 + lane;
                            const int row = q / SW, c = q % SW;
                            val[i] = *reinterpret_cast<const float4 *>(stg + ((size_t)row * SW + (c ^ (row & 7))) * 16);
                        }
                        if (mrow + 32 * P <= f.n_out) {
#pragma unroll
                            for (int i = 0; i < SW; ++i) {
                                const int q = i * 32 + lane;
                                *reinterpret_cast<float4 *>(out + mrow + (q / SW) * P + phase0 + 2 * (q % SW)) = val[i];
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < SW; ++i) {
                                const int q = i * 32 + lane;
                                const long long m = mrow + (long long)(q / SW) * P + phase0 + 2 * (q % SW);
                                if (m + 1 < f.n_out) *reinterpret_cast<float4 *>(out + m) = val[i];
                                else if (m < f.n_out) out[m] = make_float2(val[i].x, val[i].y);
                            }
                        }
                        __syncwarp();
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == UM_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

// =====================================================================================================================
// Polyphase variant for Decimate with D >= 5 (config C3: 255 taps, D = 10).  The candidate-offset kernel above spends
// its MMAs on all 32/g offsets of a row although only one in D/g is a kept output.  Here the stream is split
// into D PHASE PLANES x_p[n] = x[A0 + D n + p] (a converter lane takes 4 or 8 n x D phases = whole raw 16-byte chunks and
// emits one 8- or 16-byte piece per plane: one PRMT per output word), and
//     y[m] = sum_p sum_t h_p[t] x_p[m + t],      h_p[t] = c[K-1 - (D t + p - delta)]
// is D short unit-stride FIRs: per phase a Toeplitz MMA chain with rows 8 outputs apart (16-byte pitch, no swizzle,
// N = 48), all accumulating into the same TMEM columns, and EVERY computed output is kept.  MMA operand traffic per
// input sample drops from 33 to 16 bytes, the kept-output test disappears from the epilogue.
// =====================================================================================================================
// Staging (round 2): a loader warp brings every raw tile by ONE TMA bulk copy into a ring of linear slots, converter warps
// split a slot into the planes.  (Round 1: every producer lane cp.async'ed ITS unit's 16 D contiguous bytes so that no
// barrier was needed between the copy and the split -- a warp instruction then touched 32 different 128-byte lines, and
// that, not the MMA count, was what C3 saturated on: 1036 -> 1500 Gsamples/s, profiles/r02_ab_c3_poly.txt.)
// MEASURED AND REMOVED (round 2, each bit-identical and green on the whole FIR suite, each within 5 % of this kernel on the
// same box): window rows 16 outputs apart (32-byte pitch = SWIZZLE_32B, N = 96: the same 30 MMAs produce 2048 outputs, 36 %
// less tensor operand traffic, but 92 KB of tables leave room for two half-tile raw slots only: -5 .. -9 %; an earlier
// version without any raw ring: 930 vs 1035); I / Q byte planes (16 outputs per 16-byte row, 40 MMAs of N = 48 per 2048
// outputs, a third less operand traffic, 40 instead of 20 PRMT per converter item: equal at 2^28, -3 % at 2^26); skipping
// the last k-step of phases whose taps end earlier (27 instead of 30 MMAs: -2 %).  ncu of THIS kernel: the tensor core's
// shared-memory operand pipe is 91 % busy (44 wavefronts per MMA = 32 of A + 12 of B); with it relieved, the converters or
// the raw ring take over at the same level.
constexpr int UP_TILE_OUT = 1024;  // outputs per tile = 128 rows x 8
constexpr int UP_SETS = 4;         // accumulator sets of 48 TMEM columns
constexpr int UP_RAW = 3;          // raw ring slots: the loader runs up to 3 tiles ahead (21 KB bulk copies reach the full HBM rate from 3 slots on)
__host__ __device__ constexpr int up_ksteps(int K, int D) { return (7 + (K + 6) / D) / 16 + 1; }
__host__ __device__ constexpr int up_nsub(int KS) { return 8 * 128 + 16 * KS; }  // sub-samples per plane per tile
// Raw slots are LINEAR copies of the input (one TMA bulk copy each).  A converter lane reads whole 16-byte chunks of its
// item with LDS.128; with a lane stride of 16 D bytes (a full unit = D chunks per lane) the 8 lanes of a quarter warp
// fall on 8 / gcd(D, 8) bank groups.  For D = 2 (mod 4) (C3's D = 10) a lane takes HALF a unit instead (D / 2 chunks,
// 4 sub-samples of every phase, one 8-byte store per plane): the lane stride of 8 D bytes is an odd multiple of 16 and
// every quarter warp is conflict free.  (Round 1 skewed the slot instead; a bulk copy cannot skew.)
__host__ __device__ constexpr bool up_half(int D) { return D % 4 == 2; }
__host__ __device__ constexpr size_t up_raw_bytes(int D, int KS) { return (size_t)D * 2 * up_nsub(KS); }
__host__ __device__ constexpr size_t up_smem_bytes(int D, int KS, int stages) {
    // stages of D planes + tables + raw ring (UP_RAW slots) + 1 KB slack + barriers
    return (size_t)stages * D * 2 * up_nsub(KS) + UP_RAW * up_raw_bytes(D, KS) + (size_t)D * KS * 48 * 32 + 1024 + 256;
}

// roles: 9 converter warps (the phase split; 268 half units per tile at D = 10), 1 loader warp, 2 MMA warps taking
// alternate tiles, 8 epilogue warps (warp % 4 = TMEM lane quarter)
constexpr int UP_CONV_WARPS = 9, UP_LOAD_WARP = UP_CONV_WARPS, UP_MMA_WARP = UP_CONV_WARPS + 1, UP_MMA_WARPS = 2,
              UP_EPI_WARP0 = UP_MMA_WARP + UP_MMA_WARPS, UP_THREADS = (UP_EPI_WARP0 + 8) * 32;
static_assert(UP_EPI_WARP0 % 4 == 0, "epilogue warps must start on a TMEM lane-quarter boundary");

// all D * KS MMAs of a tile, fully unrolled: A descriptor = plane p (PLB / 16 = 128 + 2 KS descriptor units apart) + 2 kk,
// B descriptor = block p * KS + kk of the table (48 x 32 B = 96 units)
template <int D, int KS>
__device__ __forceinline__ void up_issue_tile(uint32_t d0, uint64_t ap, uint64_t bd, uint32_t idesc) {
    constexpr uint64_t PSTEP = 128 + 2 * KS, BSTEP = (48 * 32) >> 4;
    umma_i8<false>(d0, ap, bd, idesc);
#pragma unroll
    for (int j = 1; j < D * KS; ++j)
        umma_i8<true>(d0, ap + (uint64_t)(j / KS) * PSTEP + 2 * (uint64_t)(j % KS), bd + (uint64_t)j * BSTEP, idesc);
}

template <int D>
__global__ void __launch_bounds__(UP_THREADS, 1) fir_umma_poly_kernel(const UmArgs a) {
    constexpr int N = 48;
    constexpr int NCONV = 32 * UP_CONV_WARPS;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * UM_STAGES + 2 * UP_SETS + 2 * UP_RAW + 1];
    __shared__ uint32_t tmem_base_s;
    const FirArgs &f = a.f;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KS = a.KS, NST = a.stages;
    const int NSUB = up_nsub(KS), PLB = 2 * NSUB, SB = D * PLB;  // plane / stage bytes
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t stage0 = base;
    const uint32_t tab_s = stage0 + NST * SB;
    uint8_t *gen = smem_raw + (base - smem_u32(smem_raw));
    uint8_t *raw0 = gen + (size_t)NST * SB + (size_t)D * KS * N * 32;
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (UM_STAGES + s); };
    auto accf_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + s); };
    auto acce_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + UP_SETS + s); };
    auto rawfull_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + 2 * UP_SETS + s); };
    auto rawfree_bar = [&](int s) { return bar0 + 8u * (2 * UM_STAGES + 2 * UP_SETS + UP_RAW + s); };
    const uint32_t tab_bar = bar0 + 8u * (2 * UM_STAGES + 2 * UP_SETS + 2 * UP_RAW);
    if (tid == 0) {
        for (int s = 0; s < UM_STAGES; ++s) { mbar_init(full_bar(s), NCONV); mbar_init(empty_bar(s), 1); }
        for (int s = 0; s < UP_SETS; ++s) { mbar_init(accf_bar(s), 1); mbar_init(acce_bar(s), 4); }
        for (int s = 0; s < UP_RAW; ++s) { mbar_init(rawfull_bar(s), 1); mbar_init(rawfree_bar(s), UP_CONV_WARPS); }
        mbar_init(tab_bar, 1);
        mbar_init_fence();
    }
    if (warp == UP_MMA_WARP) {
        tmem_alloc<256>(smem_u32(&tmem_base_s));
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const long long nwork = (long long)a.ntiles * f.n_ch;
    const long long wstride = gridDim.x;

    if (warp == UP_LOAD_WARP) {
        // ================= loader warp: raw tiles by TMA bulk copies, UP_RAW tiles ahead =================
        // Round 1 gave every lane ITS unit's 16 D contiguous bytes as D 16-byte cp.async: a warp instruction then
        // touches 32 different 128-byte lines (lane stride 16 D bytes), i.e. 32 L1 tag passes for 512 bytes.  Here the
        // copy engine moves the tile: ONE bulk copy into a linear slot.  (One copy per skew group of 8 / gcd(D, 8) units,
        // which keeps the conflict-free skewed layout, was measured far slower: 34 copies of 640 bytes per tile.)
        const int nunits = NSUB / 8;
        const int RAWB = (int)up_raw_bytes(D, KS);
        long long it = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride, ++it) {
            const int slot = (int)(it % UP_RAW);
            if (it >= UP_RAW) mbar_wait(rawfree_bar(slot), (uint32_t)((it / UP_RAW - 1) & 1));
            int ch; long long wt;
            split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
            const long long w0 = f.first - (f.K - 1) - a.delta + wt * (long long)(UP_TILE_OUT * D);
            const unsigned char *in = (const unsigned char *)f.in + (long long)ch * f.in_stride * 2;
            uint8_t *rs = raw0 + (size_t)slot * RAWB;
            const uint32_t rs_s = smem_u32(rs);
            // chunks [q_lo, q_hi) of the tile are whole, in-range 16-byte pieces of the input: ONE bulk copy.  The rest
            // (first / last tile of a channel: carried history, "zero" = byte 128, ragged end) by plain stores.
            const int nq = nunits * D;
            long long ql = w0 >= 0 ? 0 : (-w0 + 7) / 8, qh = (f.n_in - w0) / 8;
            const int q_lo = (int)min(ql, (long long)nq), q_hi = (int)max(min(qh, (long long)nq), (long long)q_lo);
            const uint32_t bytes = 16u * (uint32_t)(q_hi - q_lo);
            if (q_lo > 0 || q_hi < nq) {
                const unsigned char *hist = (const unsigned char *)f.hist + (long long)ch * f.hist_stride * 2;
                for (int q = lane; q < nq - (q_hi - q_lo); q += 32) {
                    const int qq = q < q_lo ? q : q + (q_hi - q_lo);
                    const long long s0 = w0 + 8LL * qq;
                    if (s0 < f.n_in) {
                        unsigned short h[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const long long s = s0 + i;
                            unsigned short x = 0x8080;
                            if (s >= 0) { if (s < f.n_in) x = *reinterpret_cast<const unsigned short *>(in + 2 * s); }
                            else if (s >= -(long long)f.HL) x = *reinterpret_cast<const unsigned short *>(hist + 2 * ((long long)f.HL + s));
                            h[i] = x;
                        }
                        uint4 qv;
                        qv.x = h[0] | ((unsigned)h[1] << 16); qv.y = h[2] | ((unsigned)h[3] << 16);
                        qv.z = h[4] | ((unsigned)h[5] << 16); qv.w = h[6] | ((unsigned)h[7] << 16);
                        *reinterpret_cast<uint4 *>(rs + 16 * qq) = qv;
                    }
                }
                __syncwarp();
            }
            if (lane == 0) {
                if (bytes) {
                    mbar_arrive_expect_tx(rawfull_bar(slot), bytes);
                    tma_bulk_g2s(rs_s + 16u * (uint32_t)q_lo, in + 2 * (w0 + 8LL * q_lo), bytes, rawfull_bar(slot));
                } else {
                    mbar_arrive(rawfull_bar(slot));
                }
            }
        }
    } else if (warp < UP_CONV_WARPS) {
        // ================= converters: raw slot -> D phase planes =================
        const int ptid = warp * 32 + lane;
        constexpr bool HALF = up_half(D);
        constexpr int CH = HALF ? D / 2 : D;    // 16-byte chunks per item
        constexpr int NW = HALF ? 2 : 4;        // output words per plane per item
        const int nitems = (NSUB / 8) * (HALF ? 2 : 1);
        const int RAWB = (int)up_raw_bytes(D, KS);
        int stage = 0, slot = 0;
        uint32_t ph = 0, rph = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride) {
            mbar_wait(rawfull_bar(slot), rph);
            mbar_wait(empty_bar(stage), ph ^ 1u);
            uint8_t *st_g = gen + (size_t)stage * SB;
            const uint8_t *rs = raw0 + (size_t)slot * RAWB;
            for (int i = ptid; i < nitems; i += NCONV) {
                uint32_t rw[4 * CH];  // the item's samples, 2 per word (I, Q bytes of a sample stay together)
#pragma unroll
                for (int c = 0; c < CH; ++c) {
                    const uint4 q = *reinterpret_cast<const uint4 *>(rs + 16 * (i * CH + c));
                    rw[4 * c] = q.x; rw[4 * c + 1] = q.y; rw[4 * c + 2] = q.z; rw[4 * c + 3] = q.w;
                }
#pragma unroll
                for (int p = 0; p < D; ++p) {
                    uint32_t o[NW];
#pragma unroll
                    for (int wd = 0; wd < NW; ++wd) {
                        // plane sub-samples 2wd, 2wd+1 of this item = its raw samples D*(2wd) + p, D*(2wd+1) + p
                        // (an item starts an even number of samples into its unit: the parities are the unit's)
                        const int sa = D * (2 * wd) + p, sb = D * (2 * wd + 1) + p;
                        const uint32_t sel = (uint32_t)(2 * (sa & 1)) | ((uint32_t)(2 * (sa & 1) + 1) << 4) |
                                             ((uint32_t)(4 + 2 * (sb & 1)) << 8) | ((uint32_t)(5 + 2 * (sb & 1)) << 12);
                        o[wd] = __byte_perm(rw[sa >> 1], rw[sb >> 1], sel);
                    }
                    if (HALF) *reinterpret_cast<uint2 *>(st_g + (size_t)p * PLB + 8 * i) = make_uint2(o[0], o[1]);
                    else *reinterpret_cast<uint4 *>(st_g + (size_t)p * PLB + 16 * i) = make_uint4(o[0], o[1], o[NW - 2], o[NW - 1]);
                }
            }
            fence_proxy_async();  // plain stores -> visible to the tensor core's (async proxy) operand reads
            mbar_arrive(full_bar(stage));
            __syncwarp();
            if (lane == 0) mbar_arrive(rawfree_bar(slot));  // this warp's reads of the slot are done
            if (++stage == NST) { stage = 0; ph ^= 1u; }
            if (++slot == UP_RAW) { slot = 0; rph ^= 1u; }
        }
    } else if (warp < UP_EPI_WARP0) {
        // ================= MMA issuers: warp j takes tiles j, j + 2, ...; D phases x KS k-steps into one set =================
        const int mw = warp - UP_MMA_WARP;
        const uint32_t idesc = idesc_u8s8_s32(128, N);
        const uint64_t bdesc0 = smem_desc(tab_s, 128, 256, 0);
        {
            // the tap tables arrive by one bulk copy while the first raw tile is loaded and converted
            if (mw == 0 && elect_one()) {
                mbar_arrive_expect_tx(tab_bar, (uint32_t)(D * KS * N * 32));
                tma_bulk_g2s(tab_s, a.tab, (uint32_t)(D * KS * N * 32), tab_bar);
            }
            __syncwarp();
            mbar_wait(tab_bar, 0);
        }
        long long it = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride, ++it) {
            if ((it & (UP_MMA_WARPS - 1)) != mw) continue;
            const int stage = (int)(it % NST), as = (int)(it & (UP_SETS - 1));
            const uint32_t ph = (uint32_t)((it / NST) & 1), aph = (uint32_t)((it / UP_SETS) & 1);
            mbar_wait(full_bar(stage), ph);
            mbar_wait(acce_bar(as), aph ^ 1u);
            tc_fence_after();
            if (elect_one()) {
                const uint64_t ap = smem_desc(stage0 + (uint32_t)stage * SB, 16, 128, 0);  // plane 0
                const uint32_t d0 = tmem + (uint32_t)(as * N);
                // KS is a run-time value; a loop over it made ptxas emit a dependent chain of ~12 uniform-datapath
                // instructions per MMA (ncu: the two issuing warps were busy 86 % of the time, ~145 cycles per MMA, with
                // the tensor pipe 40 % active).  Dispatch to straight-line code per KS instead: every descriptor is the
                // tile's base plus an immediate.
                switch (KS) {
                    case 1: up_issue_tile<D, 1>(d0, ap, bdesc0, idesc); break;
                    case 2: up_issue_tile<D, 2>(d0, ap, bdesc0, idesc); break;
                    case 3: up_issue_tile<D, 3>(d0, ap, bdesc0, idesc); break;
                    case 4: up_issue_tile<D, 4>(d0, ap, bdesc0, idesc); break;
                    case 5: up_issue_tile<D, 5>(d0, ap, bdesc0, idesc); break;
                    case 6: up_issue_tile<D, 6>(d0, ap, bdesc0, idesc); break;
                    default: up_issue_tile<D, 7>(d0, ap, bdesc0, idesc); break;
                }
                umma_commit(empty_bar(stage));
                umma_commit(accf_bar(as));
            }
            __syncwarp();
        }
    } else {
        // ================= epilogue: warpgroup wg takes every 4th tile, accumulator set wg =================
        const int ew = warp - UP_EPI_WARP0, wg = ew >> 2, quad = warp & 3;  // warpgroup wg: sets wg, wg + 2
        const float sc0 = a.sc[0], sc2 = a.sc[2];
        const int c10[2] = {a.magic[0][0], a.magic[1][0]}, m2[2] = {a.magic[0][2], a.magic[1][2]};
        uint32_t aph = 0;
        long long it = 0;
        for (long long w = blockIdx.x; w < nwork; w += wstride, ++it) {
            if ((it & 1) != wg) continue;
            const int set = (int)(it & (UP_SETS - 1));
            int ch; long long wt;
            split_work(w, a.ntiles, (int)f.n_ch, ch, wt);
            const long long m0 = wt * (long long)UP_TILE_OUT;
            float2 *out = (float2 *)f.out + (long long)ch * f.out_stride;
            mbar_wait(accf_bar(set), aph);
            if (set >= 2) aph ^= 1u;  // this warpgroup's two sets alternate; the parity flips after both were used
            tc_fence_after();
            uint32_t e[2][3][8];
            const uint32_t col = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(set * N);
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int dg = 0; dg < 3; ++dg) tmem_ld_16x256b_x2(col + ((uint32_t)(16 * hh) << 16) + dg * 16, e[hh][dg]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acce_bar(set));
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int cg = 0; cg < 2; ++cg)
#pragma unroll
                    for (int rs = 0; rs < 2; ++rs) {
                        const int i0 = 4 * cg + 2 * rs;
                        const long long m = m0 + 8 * (quad * 32 + 16 * hh + 8 * rs + (lane >> 2)) + 4 * cg + (lane & 3);
                        if (m < f.n_out) {
                            const float fI = (float)((int)(e[hh][1][i0] << 8) + (int)e[hh][0][i0] + c10[0]);
                            const float fQ = (float)((int)(e[hh][1][i0 + 1] << 8) + (int)e[hh][0][i0 + 1] + c10[1]);
                            const float gI = __int_as_float((int)e[hh][2][i0] + m2[0]) - 12582912.0f;
                            const float gQ = __int_as_float((int)e[hh][2][i0 + 1] + m2[1]) - 12582912.0f;
                            out[m] = make_float2(fmaf(gI, sc2, fI * sc0), fmaf(gQ, sc2, fQ * sc0));
                        }
                    }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == UP_MMA_WARP) {
        tc_fence_after();
        tmem_dealloc<256>(tmem);
    }
}

// balanced base-256 digits of t: t = d0 + 256 d1 + 65536 d2, d0, d1 in [-128, 127]; false if d2 leaves that range
inline bool digits3(long long t, int d[3]) {
    for (int i = 0; i < 2; ++i) {
        long long r = ((t % 256) + 256) % 256;
        if (r >= 128) r -= 256;
        d[i] = (int)r;
        t = (t - r) / 256;
    }
    d[2] = (int)t;
    return t >= -128 && t <= 127;
}

}  // namespace

static int gcd_i(int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; }

// k-steps of 16 samples: a row's window spans K + 7 (alignment) + the largest candidate offset R - g samples
int fir_umma_ksteps(int K, int R, int PC) { return (K + 7 + R - R / PC + 15) / 16; }

int fir_umma_planar_ksteps(int K, int R, int PC) { return (K + 7 + R - R / PC + 31) / 32; }

// geometry for (K, D, tap kind): row pitch R, candidates per row PC, planar (real taps) or interleaved stages;
// false if the tcgen05 path does not apply
bool fir_umma_geometry(int K, int D, bool taps_complex, bool want_planar, int *R_out, int *PC_out, int *planar_out) {
    if (K < 1 || K > UM_MAX_K || D < 1 || D > 4096) return false;
    const char *e = std::getenv("SDR_UMMA_P");
    const int forced = e ? std::atoi(e) : 0;
    *planar_out = 0;
    static const bool no_poly = std::getenv("SDR_UMMA_NO_POLY") != nullptr;  // A/B switch (tuning)
    if (!want_planar && !no_poly && (D == 5 || D == 6 || D == 7 || D == 8 || D == 9 || D == 10 || D == 12) &&
        up_smem_bytes(D, up_ksteps(K, D), 2) <= 220 * 1024) {
        *R_out = 8; *PC_out = 8; *planar_out = 2;  // polyphase planes
        return true;
    }
    if (!taps_complex && want_planar) {
        // real taps: byte planes, rows R bytes = R samples apart
        int R = 0, PC = 0;
        if (D == 1) {
            R = PC = (forced == 16) ? 16 : 32;
        } else if (64 / gcd_i(D, 64) == 16 || 64 / gcd_i(D, 64) == 32) {
            R = 64; PC = 64 / gcd_i(D, 64);
        } else if (32 / gcd_i(D, 32) == 16 || 32 / gcd_i(D, 32) == 32) {
            R = 32; PC = 32 / gcd_i(D, 32);
        }
        if (R && um_planar_smem_bytes(R, PC, fir_umma_planar_ksteps(K, R, PC), D != 1, 2) <= 220 * 1024) {
            *R_out = R; *PC_out = PC; *planar_out = 1;
            return true;
        }
    }
    if (D == 1) {
        int best = 0;
        double best_c = 1e30;
        for (int p : {8, 16, 32}) {
            const int ks = fir_umma_ksteps(K, p, p);
            if (um_smem_bytes(p, p, ks, false, 2) > 220 * 1024) continue;
            // cycles per output ~ KS * max(45, N/2) / (128 P): wide rows amortise the band padding
            const double c = (forced == p) ? 0.0 : ks * std::max(45.0, 3.0 * p) / (128.0 * p);
            if (c < best_c) { best_c = c; best = p; }
        }
        if (!best) return false;
        *R_out = *PC_out = best;
        return true;
    }
    const int g = gcd_i(D, 32);
    if (g > 4) return false;  // fewer than 8 candidates per 32-sample row: N would drop below the M = 128 minimum of 16
    const int ks = fir_umma_ksteps(K, 32, 32 / g);
    if (um_smem_bytes(32, 32 / g, ks, true, 2) > 220 * 1024) return false;
    *R_out = 32;
    *PC_out = 32 / g;
    return true;
}

// host: the 8 alignment variants of the Toeplitz tap table.  Layout [delta][kk][canonical N x 32 B block]:
// element (n, kb) of a block sits at (n/8)*256 + (kb/16)*128 + (n%8)*16 + kb%16 (no-swizzle K-major core matrices).
// Column n = digit * 2 PC + 2 u + part; candidate u is the output whose oldest sample sits g*u (+ delta) into the row.
bool fir_umma_build_tables(const float *taps, int K, bool tc, int R, int PC, int mode, int D, std::vector<uint8_t> &out, int magic[2][3], float sc[3]) {
    const bool planar = mode == 1, poly = mode == 2;
    if (K < 1 || K > UM_MAX_K || (planar && tc)) return false;
    const int KS = planar ? fir_umma_planar_ksteps(K, R, PC) : fir_umma_ksteps(K, R, PC), N = (planar ? 3 : 6) * PC, W = tc ? 2 : 1, G = R / PC;
    float cmax = 0.0f;
    for (int i = 0; i < K * W; ++i) {
        if (!std::isfinite(taps[i])) return false;
        cmax = std::fmax(cmax, std::fabs(taps[i]));
    }
    int e = 0;
    if (cmax > 0.0f) std::frexp(cmax, &e);
    int S = 23 - e;  // cmax * 2^S in [2^22, 2^23)
    std::vector<long long> t((size_t)K * W);
    for (;; --S) {
        bool ok = true;
        for (int i = 0; i < K * W && ok; ++i) {
            t[i] = std::llround(std::ldexp((double)taps[i], S));
            int d[3];
            ok = digits3(t[i], d) && digits3(-t[i], d);
        }
        if (ok) break;
    }
    // digit tables of the four roles a tap can play: +re, -im (into the I part), +im, +re (into the Q part)
    auto digit = [&](int k, int part, int q, int dg) -> int {
        long long v;
        if (!tc) v = (q == part) ? t[k] : 0;
        else if (part == 0) v = (q == 0) ? t[2 * k] : -t[2 * k + 1];
        else v = (q == 0) ? t[2 * k + 1] : t[2 * k];
        int d[3];
        digits3(v, d);
        return d[dg];
    };
    for (int part = 0; part < 2; ++part)
        for (int dg = 0; dg < 3; ++dg) {
            long long s = 0;
            for (int k = 0; k < K; ++k) s += digit(k, part, 0, dg) + digit(k, part, 1, dg);
            magic[part][dg] = (int)(128 * s);  // C_d
        }
    for (int part = 0; part < 2; ++part) {
        const long long c10 = -(256LL * magic[part][1] + magic[part][0]);
        magic[part][0] = (int)(unsigned)(unsigned long long)c10;  // two's complement wrap is what the kernel's s32 add expects
        magic[part][1] = 0;
        magic[part][2] = (int)(0x4B400000LL - magic[part][2]);
    }
    const float base = std::ldexp(1.0f, -S - 7);
    sc[0] = base; sc[1] = base * 256.0f; sc[2] = base * 65536.0f;
    if (poly) {
        // [delta][phase][kk][canonical 48 x 32 B block]: column dg*16 + 2c + part, byte kb = sub-sample kb/2 (I, Q)
        const int KSP = up_ksteps(K, D);
        out.assign((size_t)8 * D * KSP * 48 * 32, 0);
        for (int delta = 0; delta < 8; ++delta)
            for (int ph = 0; ph < D; ++ph)
                for (int kk = 0; kk < KSP; ++kk) {
                    uint8_t *blk = out.data() + (((size_t)delta * D + ph) * KSP + kk) * 48 * 32;
                    for (int n = 0; n < 48; ++n) {
                        const int dg = n / 16, c = (n % 16) / 2, part = n & 1;
                        for (int kb = 0; kb < 32; ++kb) {
                            const int kap = kk * 16 + kb / 2, q = kb & 1;
                            const int t = kap - c, j = D * t + ph - delta;  // raw offset of this sub-sample from the window start
                            int v = 0;
                            if (t >= 0 && j >= 0 && j < K) v = digit(K - 1 - j, part, q, dg);
                            blk[(n / 8) * 256 + (kb / 16) * 128 + (n % 8) * 16 + kb % 16] = (uint8_t)(int8_t)v;
                        }
                    }
                }
        return true;
    }
    out.assign((size_t)8 * KS * N * 32, 0);
    for (int delta = 0; delta < 8; ++delta)
        for (int kk = 0; kk < KS; ++kk) {
            uint8_t *blk = out.data() + ((size_t)delta * KS + kk) * N * 32;
            for (int n = 0; n < N; ++n) {
                // interleaved: column (digit, candidate, part), byte kb = sample kb/2, part kb&1
                // planar:      column (digit, candidate),       byte kb = sample kb of the plane
                const int dg = planar ? n / PC : n / (2 * PC), u = planar ? n % PC : (n % (2 * PC)) / 2, part = planar ? 0 : (n & 1);
                for (int kb = 0; kb < 32; ++kb) {
                    const int s = planar ? kk * 32 + kb : kk * 16 + kb / 2, q = planar ? 0 : (kb & 1);
                    const int k = K - 1 + delta + G * u - s;
                    int v = 0;
                    if (k >= 0 && k < K) v = digit(k, part, q, dg);
                    blk[(n / 8) * 256 + (kb / 16) * 128 + (n % 8) * 16 + kb % 16] = (uint8_t)(int8_t)v;
                }
            }
        }
    return true;
}

// returns SDR_ERR_UNSUPPORTED when this path does not apply (caller falls back to the mma.sync / CUDA-core kernels)
static int fir_umma_poly_launch(const FirArgs &f, const uint8_t *d_tables, const int magic[2][3], const float sc[3], cudaStream_t st) {
    const int D = f.D, KS = up_ksteps(f.K, D);
    int stages = UM_STAGES;
    while (stages > 2 && up_smem_bytes(D, KS, stages) > 222 * 1024) --stages;
    const size_t smem = up_smem_bytes(D, KS, stages);
    if (smem > 222 * 1024) return SDR_ERR_UNSUPPORTED;
    UmArgs a;
    a.f = f;
    a.KS = KS;
    a.stages = stages;
    // the window start in + 2 (first - (K-1) - delta) must be 16-byte aligned for the 16-byte copies: delta absorbs
    // both the position of the first needed sample and the alignment of the caller's pointer (any even address)
    long long d = (f.first - (f.K - 1) + (long long)(((uintptr_t)f.in & 15) >> 1)) % 8;
    if (d < 0) d += 8;
    a.delta = (int)d;
    a.tab = d_tables + (size_t)d * D * KS * 48 * 32;
    a.stage_bytes = D * 2 * up_nsub(KS);
    a.n_rows = 0;
    a.dmagic = 0;
    a.ntiles = (int)((f.n_out + UP_TILE_OUT - 1) / UP_TILE_OUT);
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 3; ++j) a.magic[i][j] = magic[i][j];
    for (int j = 0; j < 3; ++j) a.sc[j] = sc[j];
    const int sms = current_sm_count();
    const long long nwork = (long long)a.ntiles * f.n_ch;
    const unsigned grid = (unsigned)std::min<long long>(nwork, sms);
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kern<<<grid, UP_THREADS, smem, st>>>(a);
        count_launch();
        return launch_status();
    };
    switch (D) {
        case 5: return go(fir_umma_poly_kernel<5>);
        case 6: return go(fir_umma_poly_kernel<6>);
        case 7: return go(fir_umma_poly_kernel<7>);
        case 8: return go(fir_umma_poly_kernel<8>);
        case 9: return go(fir_umma_poly_kernel<9>);
        case 10: return go(fir_umma_poly_kernel<10>);
        case 12: return go(fir_umma_poly_kernel<12>);
    }
    return SDR_ERR_UNSUPPORTED;
}

// Tensor map over the raw byte stream for fir_umma_kernel's stages: {ROWB bytes, ROWB/16 sub-offsets (stride 16 B),
// rows (stride ROWB)[, channels (stride 2 in_stride)]}, box {ROWB, 1, rows, 1}, swizzle = the A descriptor's.  Returns
// false when TMA cannot serve this call (the kernel then stages with cp.async, same bytes in the same places).
static bool um_make_tensor_map(const FirArgs &f, int R, int nchunks, int stage_bytes, UmArgs &a, CUtensorMap *tm) {
    // MEASURED (round 2, A/B on one box, profiles/r02_ab_tma.txt): with 64-byte box rows at 16-byte sub-offsets the tensor
    // copy is 4-5 % SLOWER than the three LDGSTS producer warps on the HBM-bound 64-tap configs (C1 457-461 vs 482-487,
    // complex taps 447-455 vs 467-473 Gsamples/s) and equal on the tensor-bound 255-tap one (311 vs 312).  The stage layout
    // forces small rows (the window rows' pitch IS the swizzle width), and a 1-D bulk copy cannot swizzle.  So this
    // kernel keeps cp.async by default and takes the TMA path with SDR_UMMA_TMA=1 (same bytes in the same places:
    // test_tcgen05_tma_staging_gives_the_same_bits); the c64 FIR and the 1024-point FFT, whose stages are plain linear
    // copies, use TMA bulk copies unconditionally.
    static const bool on = std::getenv("SDR_UMMA_TMA") != nullptr;
    EncodeTiledFn enc = encode_tiled_fn();
    if (!on || !enc) return false;
    const int W = 2 * R;
    const uintptr_t addr = (uintptr_t)f.in;
    const int shift = (int)(addr & 15);
    const long long nbytes = 2 * f.n_in + shift;
    const long long rows_total = (nbytes - (W - 16)) / W;
    if (rows_total < 1) return false;
    const int need_rows = (16 * nchunks + W - 1) / W;
    const int nbox = (need_rows + 255) / 256;
    int rows = ((need_rows + nbox - 1) / nbox + 7) & ~7;  // multiples of 8 rows keep the swizzle period between boxes
    if (rows > 256 || (long long)nbox * rows * W > stage_bytes) return false;
    const bool multi = f.n_ch > 1;
    if (multi && ((2 * f.in_stride) % 16 != 0 || 2 * f.in_stride >= (1LL << 40))) return false;
    cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)(W / 16), (cuuint64_t)rows_total, (cuuint64_t)f.n_ch};
    cuuint64_t strides[3] = {16, (cuuint64_t)W, (cuuint64_t)(2 * f.in_stride)};  // bytes, dims 1..3
    cuuint32_t box[4] = {(cuuint32_t)W, 1, (cuuint32_t)rows, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUtensorMapSwizzle sw = R == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : R == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, multi ? 4 : 3, (void *)(addr - shift), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    a.use_tma = 1;
    a.tma_rows = rows;
    a.tma_nbox = nbox;
    a.tma_shift = shift;
    a.tma_need = need_rows + 1;  // + 1: a window that starts at a 16-byte sub-offset spills into one more row
    a.tma_rows_total = rows_total;
    return true;
}

int fir_umma_launch(const FirArgs &f, int R, int PC, int mode, const uint8_t *d_tables, const int magic[2][3], const float sc[3], cudaStream_t st) {
    const bool planar = mode == 1;
    if (f.n_out <= 0) return SDR_OK;
    if (mode == 2) {
        if (f.K > UM_MAX_K || ((uintptr_t)f.in & 1) || ((uintptr_t)f.out & 7) || ((uintptr_t)f.hist & 1) || (f.n_ch > 1 && (f.in_stride & 7)))
            return SDR_ERR_UNSUPPORTED;
        return fir_umma_poly_launch(f, d_tables, magic, sc, st);
    }
    if (f.K > UM_MAX_K || (f.D == 1 && R != PC) || (f.D != 1 && !planar && R != 32)) return SDR_ERR_UNSUPPORTED;
    // rows of a multi-channel call must keep the alignment (mod 16 bytes) of the first one (strides are ignored for one
    // channel); the input itself may start at any even address: the kernel family gives the SAME bits for every
    // alignment and blocking, which is what lets a stream be cut across GPUs at arbitrary multiples of D
    if (((uintptr_t)f.in & 1) || ((uintptr_t)f.out & (planar ? 15 : 7)) || ((uintptr_t)f.hist & 1) ||
        (f.n_ch > 1 && ((planar && (f.out_stride & 1)) || (f.in_stride & 7))))
        return SDR_ERR_UNSUPPORTED;
    const bool dec = f.D != 1;
    const int KS = planar ? fir_umma_planar_ksteps(f.K, R, PC) : fir_umma_ksteps(f.K, R, PC);
    auto smem_of = [&](int st_) { return planar ? um_planar_smem_bytes(R, PC, KS, dec, st_) : um_smem_bytes(R, PC, KS, dec, st_); };
    int stages = UM_STAGES;
    while (stages > 2 && smem_of(stages) > 220 * 1024) --stages;
    const size_t smem = smem_of(stages);
    if (smem > 220 * 1024) return SDR_ERR_UNSUPPORTED;
    UmArgs a;
    a.stages = stages;
    a.f = f;
    a.KS = KS;
    long long d = (f.first - (f.K - 1) + (long long)(((uintptr_t)f.in & 15) >> 1)) % 8;  // see fir_umma_poly_launch
    if (d < 0) d += 8;
    a.delta = (int)d;
    a.tab = d_tables + (size_t)d * KS * (planar ? 3 : 6) * PC * 32;
    a.stage_bytes = planar ? 2 * um_plane_bytes(R, PC, KS) : um_stage_bytes(R, PC, KS);
    a.n_rows = ((f.n_out - 1) * (long long)f.D) / R + 1;
    const int tile_rows = 128 * (32 / PC);
    a.ntiles = (int)((a.n_rows + tile_rows - 1) / tile_rows);
    a.dmagic = (unsigned)((1ull << 32) / (unsigned long long)f.D + 1ull);
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 3; ++j) a.magic[i][j] = magic[i][j];
    for (int j = 0; j < 3; ++j) a.sc[j] = sc[j];
    const int sms = current_sm_count();
    const long long nwork = (long long)a.ntiles * f.n_ch;
    const unsigned grid = (unsigned)std::min<long long>(nwork, sms);
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kern<<<grid, UM_THREADS, smem, st>>>(a);
        count_launch();
        return launch_status();
    };
    // interleaved-bytes kernel: stages through TMA when a tensor map can be built for this call
    CUtensorMap tm;
    std::memset(&tm, 0, sizeof(tm));
    if (!planar) {
        const int MB = 32 / PC, ROWB = 2 * R;
        const int nchunks = (ROWB * (128 * MB - 1) + 32 * KS + 15) / 16;
        um_make_tensor_map(f, R, nchunks, a.stage_bytes, a, &tm);
    }
    auto go_tm = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kern<<<grid, UM_THREADS, smem, st>>>(a, tm);
        count_launch();
        return launch_status();
    };
    if (planar) {
        if (!dec && R == 16) return go(fir_umma_planar_kernel<16, 16, false>);
        if (!dec && R == 32) return go(fir_umma_planar_kernel<32, 32, false>);
        if (dec && R == 64 && PC == 16) return go(fir_umma_planar_kernel<64, 16, true>);
        if (dec && R == 64 && PC == 32) return go(fir_umma_planar_kernel<64, 32, true>);
        if (dec && R == 32 && PC == 16) return go(fir_umma_planar_kernel<32, 16, true>);
        if (dec && R == 32 && PC == 32) return go(fir_umma_planar_kernel<32, 32, true>);
        return SDR_ERR_UNSUPPORTED;
    }
    if (!dec) {
        switch (R) {
            case 8: return go_tm(fir_umma_kernel<8, 8, false>);
            case 16: return go_tm(fir_umma_kernel<16, 16, false>);
            case 32: return go_tm(fir_umma_kernel<32, 32, false>);
        }
    } else if (R == 32) {
        switch (PC) {
            case 8: return go_tm(fir_umma_kernel<32, 8, true>);
            case 16: return go_tm(fir_umma_kernel<32, 16, true>);
            case 32: return go_tm(fir_umma_kernel<32, 32, true>);
        }
    }
    return SDR_ERR_UNSUPPORTED;
}

}  // namespace sdr

// pll.cu -- K4: batched PLL, one lane per independent stream (the loop is a recurrence:
// the NCO value computed at sample n is an input of sample n+1, src/filter/pll.rs:70-76).
//
// Replaces Pll::apply (src/filter/pll.rs:70-85) with its Biquad sub-filters
// (src/filter/biquad.rs:43-56) for n_streams streams at once.
//
// Every f32 operation is issued in the reference's order with explicit _rn intrinsics so the
// compiler cannot contract mul+add into FMA (rustc never does).  The three transcendental calls
// (atan2, cos, sin) are the only place where results can differ from the host libm:
//   default          : own branch-free f32 routines within ~1 ulp of libm's atan2f / sinf / cosf, arranged for the depth
//                      and the instruction count of the dependent chain (219 cycles per sample)
//   SDR_PLL_F64_MATH : evaluated in f64 (~1e-12) and rounded to f32: differs from a correctly rounded libm only at rare
//                      near-ties (455 cycles per sample)
// Both track the CPU oracle to the same bars (tests/test_gpu_pll_resample.py).
// Data movement: a warp moves [32 streams x 32 samples] tiles between HBM and shared memory with
// 256-byte row segments, so the lane-per-stream inner loop reads shared memory, not strided HBM.
#include "kernels.h"
#include "ptx.cuh"

namespace sdr {

namespace {

constexpr float PI_F = 3.14159265358979323846f;
constexpr int PLL_CHUNK = 32;  // samples per staged tile

struct Biquad1 {
    float b0, b1, b2, na1, na2;
    int kind;
};

// GEN = false: the caller knows the filter is not filter::Identity (no kind test on the dependent chain)
template <bool GEN = true>
__device__ __forceinline__ float bq_apply(const Biquad1 &c, float v, float &x1, float &x2, float &y1, float &y2) {
    if (GEN && c.kind == SDR_BQ_IDENTITY) return v;
    // out = 0; out += v*b0; out += x1*b1; out += x2*b2; out += y1*na1; out += y2*na2  (biquad.rs:44-49)
    float out = __fadd_rn(0.0f, __fmul_rn(v, c.b0));
    out = __fadd_rn(out, __fmul_rn(x1, c.b1));
    out = __fadd_rn(out, __fmul_rn(x2, c.b2));
    out = __fadd_rn(out, __fmul_rn(y1, c.na1));
    out = __fadd_rn(out, __fmul_rn(y2, c.na2));
    x2 = x1; x1 = v;
    y2 = y1; y1 = out;
    return out;
}

// ---- branch-free atan2 / sincos -------------------------------------------------------------------------------------
// Two sets: f32 routines within ~1 ulp (default) and, with SDR_PLL_F64_MATH, f64 evaluation rounded to f32 (the f32
// results are then the correctly rounded ones except for ~1e-4 of the arguments, like the f64 libm calls they replace).
// The PLL is one dependent chain per stream on a single warp, so what matters is the DEPTH of these routines and their
// instruction count: no slow-path branches, one reciprocal, Estrin-evaluated polynomials.

// f64 quotient for the atan2 below, 0 < den < 1e300 (f32 magnitudes widened to f64: no rescaling needed): the
// 20-bit hardware seed (MUFU.RCP64H, no f32 round trip) and ONE Newton step give 2^-40 -- the result is rounded to f32
// afterwards, a correctly rounded f64 division would buy nothing.  Depth: MUFU + 2 DFMA + DMUL (was 3 F2F + MUFU + 7).
__device__ __forceinline__ double div_fast64(double num, double den) {
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(den));
    const double e = __fma_rn(-den, r0, 1.0);
    const double r1 = __fma_rn(r0, e, r0);
    return num * r1;
}

// The f64 routine on the PLL's dependent chain, arranged for DEPTH (a dependent DFMA costs ~18 cycles here):
//   * the same octant reduction, but the three fix-ups (pi/4 + r, pi/2 - r, pi - r, -r) are folded into ONE
//     fma(S, r, C): S = +-1 and C come from the operand signs and magnitudes, off the chain;
//   * division by seed + one Newton step (div_fast64);
//   * atan(t) = t + t z A(z) with an 8-term near-minimax A on z <= tan^2(pi/8) (Chebyshev-node fit, relative error
//     1.1e-13 -- the f32 result is still the correctly rounded one except for ~2e-6 of the arguments), Estrin in 3 levels
//     instead of the 14-term Taylor polynomial's 4.
__device__ __forceinline__ double atan2_f64(float yf, float xf) {
    // magnitudes ordered in f32 (one FMNMX each; widening is exact and monotone, so the f64 values are the same)
    const float axf = fabsf(xf), ayf = fabsf(yf);
    const float mxf = fmaxf(axf, ayf), mnf = fminf(axf, ayf);
    const double mx = (double)mxf, mn = (double)mnf;
    // which side of tan(pi/8) is decided in f32 too: an argument within an ulp of the boundary may take either branch,
    // both are accurate there (the polynomial's error stays below 2e-13 for z up to 0.1716 * (1 + 1e-6))
    const bool red = mnf > 0.41421357f * mxf;
    const bool swap = ayf > axf, xneg = __float_as_int(xf) < 0, yneg = __float_as_int(yf) < 0;
    double C = red ? 0.78539816339744831 : 0.0, S = 1.0;
    if (swap) { C = 1.5707963267948966 - C; S = -S; }
    if (xneg) { C = 3.1415926535897932 - C; S = -S; }
    if (yneg) { C = -C; S = -S; }
    const double num = red ? mn - mx : mn;
    const double den = red ? mn + mx : mx;
    const bool ok = den > 0.0 && den < 1e300;  // 0/0 -> 0 as before; inf or NaN operands must not poison the loop
    const double t = ok ? div_fast64(num, den) : 0.0;
    const double z = t * t, z2 = z * z, z4 = z2 * z2, tz = t * z;
    const double a0 = -0.33333333333266202, a1 = 0.19999999949854971, a2 = -0.14285708110368922,
                 a3 = 0.11110819716945537, a4 = -0.090841018978842836, a5 = 0.076048000638505017,
                 a6 = -0.060273075254674978, a7 = 0.032956796366944874;
    const double p0 = __fma_rn(a1, z, a0), p1 = __fma_rn(a3, z, a2), p2 = __fma_rn(a5, z, a4), p3 = __fma_rn(a7, z, a6);
    const double q0 = __fma_rn(p1, z2, p0), q1 = __fma_rn(p3, z2, p2);
    const double A = __fma_rn(q1, z4, q0);
    const double r = __fma_rn(tz, A, t);
    return __fma_rn(S, r, C);
}

// sin and cos of an f32 argument |x| < ~100 (here |x| < 2 pi) in f64: one-constant reduction by pi/2 (|k| <= 64: the dropped
// 6e-17 * k is far below the 1e-10 the f32 result needs), 4-term near-minimax polynomials in 2 Estrin levels (sin: relative
// error 1.9e-11, cos: absolute 1.9e-10 on |r| <= pi/4)
__device__ __forceinline__ void sincos_f64(float xf, double &sn, double &cs) {
    const float kf = rintf(xf * 0.63661977236758134f);
    const int q = (int)kf;
    const double k = (double)kf;
    const double r = __fma_rn(-k, 1.5707963267948966, (double)xf);
    const double s = r * r, s2 = s * s, rs = r * s;
    const double S = __fma_rn(__fma_rn(2.7249925803001736e-06, s, -0.00019840086735384028), s2,
                              __fma_rn(0.0083333318747102047, s, -0.1666666666385529));
    const double Cc = __fma_rn(__fma_rn(2.4463788293291526e-05, s, -0.001388758915560089), s2,
                               __fma_rn(0.041666650644517043, s, -0.49999999969119313));
    const double sr = __fma_rn(rs, S, r), cr = __fma_rn(s, Cc, 1.0);
    const double a = (q & 1) ? cr : sr, b = (q & 1) ? sr : cr;
    sn = (q & 2) ? -a : a;
    cs = ((q + 1) & 2) ? -b : b;
}

// ---- f32 routines arranged for DEPTH (round 2) -------------------------------------------------------------------
// The recurrence is one dependent chain per stream, so only the depth of these counts.  Both are accurate to ~1 ulp
// (the oracle calls glibc's atan2f / sinf / cosf, themselves within an ulp); tests/test_gpu_pll_resample.py holds the
// resulting trajectories to the same bars as the f64 routines above (measured: max 3.2e-6 / median 2.0e-7 of full
// scale against 3.6e-6 / 1.4e-7 -- a last-bit difference in arg or in the NCO is far below one ulp of the f32 phase
// accumulator it is added to).
//   atan2: |y|, |x| ordered by two FMNMX; t = mn / mx by MUFU.RCP + one Newton step; atan(t) = t + t z A(z), z = t^2 in
//          [0, 1], A of degree 8 (near-minimax), Estrin; the octant fix-ups are one fma(S, r, C), S = +-1 and C from the
//          operand signs, off the chain.  Against f64 atan2 on 2e6 random arguments (numpy model of the same operations,
//          rcp.approx perturbed by +-1 ulp): mean 0.37 ulp, 0.5 % of the results beyond 1 ulp, max 1.8.
//   sincos: k = rint(x * 2/pi) by the 1.5 * 2^23 magic number (no FRND / F2I on the chain), two-constant Cody-Waite,
//          degree-3 near-minimax polynomials in s = r^2 for (sin r / r - 1) / s and (cos r - 1) / s (errors 7e-11,
//          3.4e-10), Estrin in 2 levels, quadrant from the low bits of the biased float, sign by XOR.
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float div_nr(float num, float den) {  // den in [2^-100, 2^100]: seed + one Newton step
    const float r0 = rcp_approx(den);
    const float q0 = num * r0;
    return __fmaf_rn(__fmaf_rn(-den, q0, num), r0, q0);
}
__device__ __forceinline__ float atan2_fast(float yf, float xf) {
    const float axf = fabsf(xf), ayf = fabsf(yf);
    const float mx = fmaxf(axf, ayf), mn = fminf(axf, ayf);
    const bool swap = ayf > axf, xneg = __float_as_int(xf) < 0, yneg = __float_as_int(yf) < 0;
    float C = 0.0f, S = 1.0f;
    if (swap) { C = 1.5707963267948966f; S = -S; }
    if (xneg) { C = 3.1415926535897932f - C; S = -S; }
    if (yneg) { C = -C; S = -S; }
    // t = mn / mx in [0, 1]: the reciprocal is issued straight behind the FMNMX (a tan(pi/8) reduction would put a
    // compare and two selects in front of it -- measured: 2 operations more on the chain for one polynomial level
    // less).  No range branch: the divisor is clamped from below (0 / 0 -> 0, as atan2(+-0, +-0) needs); magnitudes beyond
    // 2^126, where rcp.approx.ftz flushes to zero, are not supported by this routine (the products of pll.rs:71 overflow
    // there anyway), NaN propagates as it does in the reference.
    const float t = div_nr(mn, fmaxf(mx, 1e-37f));
    // atan(t) = t + t z A(z), z = t^2 in [0, 1], A of degree 8 (near-minimax, relative error of atan 1.5e-8), Estrin
    const float z = t * t, z2 = z * z, z4 = z2 * z2, z8 = z4 * z4, tz = t * z;
    const float p01 = __fmaf_rn(0.19999796152114868f, z, -0.3333333134651184f);
    const float p23 = __fmaf_rn(0.11042594909667969f, z, -0.14279702305793762f);
    const float p45 = __fmaf_rn(0.06321871280670166f, z, -0.08690944314002991f);
    const float p67 = __fmaf_rn(0.014019518159329891f, z, -0.03671013563871384f);
    const float q0 = __fmaf_rn(p23, z2, p01), q1 = __fmaf_rn(p67, z2, p45);
    const float A = __fmaf_rn(-0.0025140501093119383f, z8, __fmaf_rn(q1, z4, q0));
    const float r = __fmaf_rn(tz, A, t);
    return __fmaf_rn(S, r, C);
}
// xf = fl(2 pi f) with f = the fractional phase in (-1, 1): the quadrant k = rint(4 f) is taken from f, beside the
// multiplication that forms xf (one operation less on the chain than rint(xf * 2/pi); the two agree except within an ulp of
// a quadrant boundary, where either k leaves |r| <= pi/4 + 1e-6)
__device__ __forceinline__ void sincos_fast(float xf, float f, float &sn, float &cs) {
    const float kb = __fmaf_rn(f, 4.0f, 12582912.0f);
    const float kf = kb - 12582912.0f;
    const int q = __float_as_int(kb);  // low two bits = k mod 4
    float r = __fmaf_rn(-kf, 1.57079637050628662109375f, xf);
    r = __fmaf_rn(-kf, -4.37113882867379e-8f, r);
    const float s = r * r, s2 = s * s, rs = r * s;
    const float ps = __fmaf_rn(__fmaf_rn(2.7417770525062224e-06f, s, -0.00019841655739583075f), s2,
                               __fmaf_rn(0.008333335630595684f, s, -0.1666666716337204f));
    const float pc = __fmaf_rn(__fmaf_rn(2.4507638954673894e-05f, s, -0.0013888041721656919f), s2,
                               __fmaf_rn(0.0416666641831398f, s, -0.5f));
    const float sr = __fmaf_rn(rs, ps, r), cr = __fmaf_rn(s, pc, 1.0f);
    const float a = (q & 1) ? cr : sr, b = (q & 1) ? sr : cr;
    sn = __int_as_float(__float_as_int(a) ^ ((q & 2) << 30));
    cs = __int_as_float(__float_as_int(b) ^ (((q + 1) & 2) << 30));
}

// The recurrence (pll.rs:71-76): everything the NEXT sample depends on.  Returns c.re and phasedif for the two filters
// that do not feed back (lock, output), which a helper warp applies one tile later.
template <bool FAST, bool GEN>
__device__ __forceinline__ float2 pll_step(const PllParams &p, const Biquad1 &lf, PllState &s, float xr, float xi) {
    // c = value * self.value.conj()           (pll.rs:71)   other = (vre, -vim)
    const float o_re = s.vre, o_im = -s.vim;
    const float cr = __fsub_rn(__fmul_rn(xr, o_re), __fmul_rn(xi, o_im));
    const float ci = __fadd_rn(__fmul_rn(xr, o_im), __fmul_rn(xi, o_re));
    // loopfilter.apply(c): Biquad<f32, Complex<f32>> acts on re and im independently
    const float lr = bq_apply<GEN>(lf, cr, s.lx1r, s.lx2r, s.ly1r, s.ly2r);
    const float li = bq_apply<GEN>(lf, ci, s.lx1i, s.lx2i, s.ly1i, s.ly2i);
    // phasedif = arg * gain                   (pll.rs:72)
    const float arg = FAST ? atan2_fast(li, lr) : (float)atan2_f64(li, lr);
    const float phasedif = __fmul_rn(arg, p.gain);
    // nphase += reference + phasedif; nphase = nphase.fract()      (pll.rs:73-74)
    float nph = __fadd_rn(s.nphase, __fadd_rn(p.reference, phasedif));
    float phase;
    if (FAST) {
        // fract = nph - trunc(nph): |nph| < 2 (checked per design on the host for the specialised kernel, per sample in
        // the general one), so trunc is 1, -1 or a zero with nph's sign: two compares and two selects instead of
        // FRND.TRUNC (14-21 cycles).  Same value.
        float tr = nph >= 1.0f ? 1.0f : __int_as_float(__float_as_int(nph) & (int)0x80000000);
        tr = nph <= -1.0f ? -1.0f : tr;
        if (GEN && !(fabsf(nph) < 2.0f)) {
            // (volatile: ptxas otherwise speculates the FRND above the branch)
            asm volatile("cvt.rzi.f32.f32 %0, %1;" : "=f"(tr) : "f"(nph));
        }
        nph = __fsub_rn(nph, tr);
        phase = __fmul_rn(2.0f * PI_F, nph);
    } else {
        nph = __fsub_rn(nph, truncf(nph));
        // phase = 2.0 * PI * nphase; value = from_polar(1.0, phase)     (pll.rs:75-76)
        phase = __fmul_rn(2.0f * PI_F, nph);
    }
    s.nphase = nph;
    if (FAST) {
        float sn, cs;
        sincos_fast(phase, nph, sn, cs);
        s.vre = cs;
        s.vim = sn;
    } else {
        double sn, cs;
        sincos_f64(phase, sn, cs);
        s.vre = (float)cs;
        s.vim = (float)sn;
    }
    return make_float2(cr, phasedif);
}

__device__ __forceinline__ Biquad1 make_bq(const float *c, int kind) {
    Biquad1 b;
    b.b0 = c[0]; b.b1 = c[1]; b.b2 = c[2]; b.na1 = c[3]; b.na2 = c[4];
    b.kind = kind;
    return b;
}

// A CTA of two warps owns 32 streams, one lane of each warp per stream.
//   warp 0 (main)   steps the recurrence, nothing else: per sample one shared load (prefetched) and one shared store
//   warp 1 (helper) cp.asyncs the next [32 streams x 32 samples] input tile (256-byte row segments), and for the
//                   PREVIOUS tile applies the two filters that do not feed back -- locked = lockfilter(c.re),
//                   output = outputfilter(phasedif * rate) (pll.rs:78-84) -- and writes the 128-byte output rows
// so the ~45 instructions per sample that are not on the dependent chain never delay it.  One barrier per tile.
template <bool FAST, bool GEN>
__global__ void __launch_bounds__(64) pll_kernel(const float2 *__restrict__ in, long long n, long long in_stride,
                                                 float *__restrict__ out, uint8_t *__restrict__ locked,
                                                 long long out_stride, const PllParams *__restrict__ params,
                                                 int params_shared, PllState *__restrict__ state, int n_streams) {
    __shared__ float2 s_in[2][32][PLL_CHUNK + 1];
    __shared__ float2 s_mid[2][32][PLL_CHUNK + 1];  // (c.re, phasedif) per sample
    __shared__ float s_out[32][PLL_CHUNK + 1];
    __shared__ uint8_t s_lk[32][PLL_CHUNK + 4];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int stream0 = blockIdx.x * 32;
    if (stream0 >= n_streams) return;
    const int my = stream0 + lane;
    const bool live = my < n_streams;
    PllParams p = params[params_shared ? 0 : (live ? my : stream0)];
    PllState st = state[live ? my : stream0];
    const Biquad1 lf = make_bq(p.lc, p.lk), of = make_bq(p.oc, p.ok), kf = make_bq(p.kc, p.kk);
    const int nrows = min(32, n_streams - stream0);
    const long long ntiles = (n + PLL_CHUNK - 1) / PLL_CHUNK;

    auto issue = [&](long long tile, int buf) {
        const long long base = tile * PLL_CHUNK;
        const int cnt = (int)min((long long)PLL_CHUNK, n - base);
        if (lane < cnt) {
#pragma unroll 8
            for (int r = 0; r < 32; ++r)
                if (r < nrows) cp_async8(&s_in[buf][r][lane], in + (long long)(stream0 + r) * in_stride + base + lane);
        }
        cp_async_commit();
    };

    if (role == 1) {
        issue(0, 0);
        cp_async_wait<0>();
    }
    __syncthreads();
    // iteration t: main steps tile t; helper loads tile t+1 and finishes tile t-1
    for (long long tile = 0; tile <= ntiles; ++tile) {
        const int buf = (int)(tile & 1);
        if (role == 0) {
            if (tile < ntiles && live) {
                const int cnt = (int)min((long long)PLL_CHUNK, n - tile * PLL_CHUNK);
                // running pointers (the indexed form recomputed the shared addresses with 7 instructions per sample) and
                // an unroll by 2 (the biquad state rotation becomes register renaming): the main warp is ISSUE bound, ncu
                // shows ~2 cycles per instruction with the samples spread evenly over the loop body
                const float2 *pin = &s_in[buf][lane][0];
                float2 *pmid = &s_mid[buf][lane][0];
                float2 xn = pin[0];
#pragma unroll 2
                for (int i = 0; i < cnt; ++i) {
                    const float2 x = xn;
                    xn = pin[i + 1];  // next sample's load leaves the dependent chain (the row has a pad element)
                    pmid[i] = pll_step<FAST, GEN>(p, lf, st, x.x, x.y);
                }
            }
        } else {
            if (tile + 1 < ntiles) issue(tile + 1, buf ^ 1);
            if (tile > 0) {
                const long long base = (tile - 1) * PLL_CHUNK;
                const int cnt = (int)min((long long)PLL_CHUNK, n - base);
                if (live) {
                    for (int i = 0; i < cnt; ++i) {
                        const float2 m = s_mid[buf ^ 1][lane][i];
                        const float lk = bq_apply<GEN>(kf, m.x, st.kx1, st.kx2, st.ky1, st.ky2);
                        s_out[lane][i] = bq_apply<GEN>(of, __fmul_rn(m.y, p.rate), st.ox1, st.ox2, st.oy1, st.oy2);
                        s_lk[lane][i] = lk > 0.01f ? 1 : 0;
                    }
                }
                __syncwarp();
                if (lane < cnt) {
#pragma unroll 8
                    for (int r = 0; r < 32; ++r)
                        if (r < nrows) {
                            out[(long long)(stream0 + r) * out_stride + base + lane] = s_out[r][lane];
                            locked[(long long)(stream0 + r) * out_stride + base + lane] = s_lk[r][lane];
                        }
                }
                __syncwarp();
            }
            cp_async_wait<0>();
        }
        __syncthreads();
    }
    if (live) {
        // the two warps hold disjoint parts of the carried state
        PllState *dst = state + my;
        if (role == 0) {
            dst->nphase = st.nphase; dst->vre = st.vre; dst->vim = st.vim;
            dst->lx1r = st.lx1r; dst->lx1i = st.lx1i; dst->lx2r = st.lx2r; dst->lx2i = st.lx2i;
            dst->ly1r = st.ly1r; dst->ly1i = st.ly1i; dst->ly2r = st.ly2r; dst->ly2i = st.ly2i;
        } else {
            dst->ox1 = st.ox1; dst->ox2 = st.ox2; dst->oy1 = st.oy1; dst->oy2 = st.oy2;
            dst->kx1 = st.kx1; dst->kx2 = st.kx2; dst->ky1 = st.ky1; dst->ky2 = st.ky2;
        }
    }
}

// Stand-alone Biquad stream filter (biquad.rs:40-56): one lane per real sequence, [32 sequences x 32 samples]
// tiles staged through shared memory like the PLL's.  W = 1: f32 streams; W = 2: c64 streams, lanes 2s, 2s+1 = re, im.
// in / out are NOT __restrict__: the FM chain (fm.cu) runs the de-emphasis in place, which is safe because every
// element is read once, by the lane that later writes it
__global__ void __launch_bounds__(32) biquad_kernel(const float *in, long long n, long long in_stride,
                                                    float *out, long long out_stride, int W,
                                                    const float *__restrict__ coef, const int *__restrict__ kind,
                                                    int coef_shared, float *__restrict__ state, int n_seq) {
    __shared__ float s_x[32][PLL_CHUNK + 1];
    const int lane = threadIdx.x;
    const int seq0 = blockIdx.x * 32;
    if (seq0 >= n_seq) return;
    const int my = seq0 + lane;
    const bool live = my < n_seq;
    const int cs = coef_shared ? 0 : (live ? my / W : seq0 / W);
    const Biquad1 bq = make_bq(coef + 5 * cs, kind[cs]);
    float x1 = 0.f, x2 = 0.f, y1 = 0.f, y2 = 0.f;
    if (live) { x1 = state[4 * my]; x2 = state[4 * my + 1]; y1 = state[4 * my + 2]; y2 = state[4 * my + 3]; }
    const int nrows = min(32, n_seq - seq0);
    // row r of the tile = sequence seq0 + r: stream (seq0 + r) / W, part (seq0 + r) % W
    for (long long base = 0; base < n; base += PLL_CHUNK) {
        const int cnt = (int)min((long long)PLL_CHUNK, n - base);
        if (lane < cnt)
            for (int r = 0; r < nrows; ++r) {
                const int sq = seq0 + r;
                s_x[r][lane] = in[((long long)(sq / W) * in_stride + base + lane) * W + sq % W];
            }
        __syncwarp();
        if (live)
            for (int i = 0; i < cnt; ++i) s_x[lane][i] = bq_apply(bq, s_x[lane][i], x1, x2, y1, y2);
        __syncwarp();
        if (lane < cnt)
            for (int r = 0; r < nrows; ++r) {
                const int sq = seq0 + r;
                out[((long long)(sq / W) * out_stride + base + lane) * W + sq % W] = s_x[r][lane];
            }
        __syncwarp();
    }
    if (live) { state[4 * my] = x1; state[4 * my + 1] = x2; state[4 * my + 2] = y1; state[4 * my + 3] = y2; }
}

// FM stereo decode around a pilot-tone Pll -- the closure of src/main.rs:62-71:
//     mono = v * 0.5
//     diff = Some(_) = pllpilot.apply(Complex::new(v, 0.0)) ? (v / pllpilot.value.powi(2)).re * 0.5 : 0.0
// One lane per station; the whole recurrence (loop, lock and output filters) runs in the lane, the input is real.
// powi(2) = z * z; f32 / Complex = (a*c/|z|^2, -a*d/|z|^2) (num-complex 0.2; the crate is not in the reference tree, see DESIGN.md).
// The rates here are 12.5x below the demodulator's (144 kS/s), so this kernel keeps the simple one-warp structure.
template <bool FAST>
__global__ void __launch_bounds__(32) pll_stereo_kernel(const float *__restrict__ in, long long n, long long in_stride,
                                                        float2 *__restrict__ out, long long out_stride,
                                                        const PllParams *__restrict__ params, int params_shared,
                                                        PllState *__restrict__ state, int n_streams) {
    const int my = blockIdx.x * 32 + threadIdx.x;
    if (my >= n_streams) return;
    const PllParams p = params[params_shared ? 0 : my];
    PllState st = state[my];
    const Biquad1 lf = make_bq(p.lc, p.lk), of = make_bq(p.oc, p.ok), kf = make_bq(p.kc, p.kk);
    const float *x = in + (long long)my * in_stride;
    float2 *y = out + (long long)my * out_stride;
    float vn = n > 0 ? __ldg(x) : 0.f;
    for (long long i = 0; i < n; ++i) {
        const float v = vn;
        if (i + 1 < n) vn = __ldg(x + i + 1);
        const float2 m = pll_step<FAST, true>(p, lf, st, v, 0.0f);
        const float lk = bq_apply<true>(kf, m.x, st.kx1, st.kx2, st.ky1, st.ky2);
        (void)bq_apply<true>(of, __fmul_rn(m.y, p.rate), st.ox1, st.ox2, st.oy1, st.oy2);  // state only (pll.rs:79)
        float diff = 0.0f;
        if (lk > 0.01f) {
            const float zr = __fsub_rn(__fmul_rn(st.vre, st.vre), __fmul_rn(st.vim, st.vim));
            const float zi = __fadd_rn(__fmul_rn(st.vre, st.vim), __fmul_rn(st.vim, st.vre));
            const float ns = __fadd_rn(__fmul_rn(zr, zr), __fmul_rn(zi, zi));
            diff = __fmul_rn(__fdiv_rn(__fmul_rn(v, zr), ns), 0.5f);
        }
        y[i] = make_float2(__fmul_rn(v, 0.5f), diff);
    }
    state[my] = st;
}

// FM demodulator output map of src/main.rs:49: |f| f.unwrap_or(0.0) / 75000.0
__global__ void fm_demod_map_kernel(const float *__restrict__ v, const uint8_t *__restrict__ locked, float *out,
                                    long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __fdiv_rn(locked[i] ? v[i] : 0.0f, 75000.0f);
}

// final stereo matrix of src/main.rs:76-80 on de-emphasised (mono, diff) frames: (mono + diff, mono - diff);
// blockIdx.y = station row
__global__ void fm_matrix_kernel(const float2 *__restrict__ md, long long md_stride, float2 *__restrict__ lr,
                                 long long lr_stride, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float2 a = md[blockIdx.y * md_stride + i];
        lr[blockIdx.y * lr_stride + i] = make_float2(__fadd_rn(a.x, a.y), __fsub_rn(a.x, a.y));
    }
}

}  // namespace

int pll_stereo_launch(const float *in, long long n, long long in_stride, float *out_md, long long out_stride,
                      const PllParams *params, int params_shared, PllState *state, int n_streams, bool fast_math,
                      cudaStream_t st) {
    if (n <= 0 || n_streams <= 0) return SDR_OK;
    const unsigned grid = (unsigned)((n_streams + 31) / 32);
    if (fast_math)
        pll_stereo_kernel<true><<<grid, 32, 0, st>>>(in, n, in_stride, (float2 *)out_md, out_stride, params, params_shared, state, n_streams);
    else
        pll_stereo_kernel<false><<<grid, 32, 0, st>>>(in, n, in_stride, (float2 *)out_md, out_stride, params, params_shared, state, n_streams);
    count_launch();
    return launch_status();
}

int fm_demod_map_launch(const float *v, const uint8_t *locked, float *out, long long n, cudaStream_t st) {
    if (n <= 0) return SDR_OK;
    fm_demod_map_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(v, locked, out, n);
    count_launch();
    return launch_status();
}

int fm_matrix_launch(const float *md, long long md_stride, float *lr, long long lr_stride, int rows, long long n_frames,
                     cudaStream_t st) {
    if (n_frames <= 0 || rows <= 0) return SDR_OK;
    fm_matrix_kernel<<<dim3((unsigned)((n_frames + 255) / 256), (unsigned)rows), 256, 0, st>>>(
        (const float2 *)md, md_stride, (float2 *)lr, lr_stride, n_frames);
    count_launch();
    return launch_status();
}

int biquad_launch(const float *in, long long n, long long in_stride, float *out, long long out_stride, int W,
                  const float *coef, const int *kind, int coef_shared, float *state, int n_seq, cudaStream_t st) {
    if (n <= 0 || n_seq <= 0) return SDR_OK;
    biquad_kernel<<<(unsigned)((n_seq + 31) / 32), 32, 0, st>>>(in, n, in_stride, out, out_stride, W, coef, kind,
                                                                 coef_shared, state, n_seq);
    count_launch();
    return launch_status();
}

int pll_launch(const float2 *in, long long n, long long in_stride, float *out, uint8_t *locked, long long out_stride,
               const PllParams *params, int params_shared, PllState *state, int n_streams, bool fast_math,
               bool any_identity, cudaStream_t st) {
    if (n <= 0 || n_streams <= 0) return SDR_OK;
    const unsigned grid = (unsigned)((n_streams + 31) / 32);
    auto go = [&](auto kern) { kern<<<grid, 64, 0, st>>>(in, n, in_stride, out, locked, out_stride, params, params_shared, state, n_streams); };
    if (fast_math) { if (any_identity) go(pll_kernel<true, true>); else go(pll_kernel<true, false>); }
    else { if (any_identity) go(pll_kernel<false, true>); else go(pll_kernel<false, false>); }
    count_launch();
    return launch_status();
}

}  // namespace sdr

// nco.cuh -- the 64-bit NCO shared by the down-converter bank (ddc.cu), the fast-convolution banks (fcfb.cu, fcsb.cu)
// and the up-converter bank (duc.cu; duc.cu and fcsb.cu take the conjugate of nco_rot): the exact derotation
// e^{-2 pi i phi / 2^64} on the device and the host-side f64 phase and rotated-taps helpers, plus the f64 DFT and the
// G' table builder of the two fast-convolution banks.  The f32 sincos of the PLL (pll.cu) and the carrier recovery
// bank's rotation built on it (csync.cu) live here too.
#pragma once
#include <cmath>
#include <utility>
#include <vector>

#include "common.cuh"

namespace sdr {

// e^{-2 pi i phi / 2^64} from the exact 64-bit phase (phi read as signed: one turn = 2^64)
__device__ __forceinline__ float2 nco_rot(uint64_t phi) {
    double s, c;
    sincospi((double)(long long)phi * 0x1p-63, &s, &c);
    return make_float2((float)c, (float)-s);
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

// e^{-2 pi i phi / 2^64} in f32 from sincos_fast (the carrier loop's rotation, csync.cu): f = fl(phi 2^-64) with phi
// read as signed, so f in [-1/2, 1/2] carries at most 2^-25 turn of rounding; the result is within a few 1e-7 of the
// exact rotation
__device__ __forceinline__ float2 nco_rot_fast(uint64_t phi) {
    const float f = __fmul_rn(__ll2float_rn((long long)phi), 0x1p-64f);
    float s, c;
    sincos_fast(__fmul_rn(f, 6.2831855f), f, s, c);
    return make_float2(c, -s);
}

constexpr double NCO_2PI = 6.283185307179586476925286766559;

// phase in turns, read as signed: (-1/2, 1/2]
inline double nco_turns(uint64_t phi) { return (double)(long long)phi * 0x1p-64; }

// complex taps g[j] = h[j] e^{+2 pi i (j inc mod 2^64) / 2^64}, rounded to f32 from f64 (interleaved re, im)
inline void nco_rotated_taps(const float *h, size_t L, uint64_t inc, std::vector<float> &g) {
    g.resize(2 * L);
    for (size_t j = 0; j < L; ++j) {
        const double t = NCO_2PI * nco_turns((uint64_t)j * inc);
        g[2 * j] = (float)((double)h[j] * std::cos(t));
        g[2 * j + 1] = (float)((double)h[j] * std::sin(t));
    }
}

// The fast-convolution banks (fcfb.cu, fcsb.cu) share their block geometry and their spectral tables.

// iterative radix-2 f64 DFT in place, re.size() a power of two: X[r] = sum_t a[t] e^{-2 pi i r t / n}
inline void fft_f64(std::vector<double> &re, std::vector<double> &im) {
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
    }
    std::vector<double> wc(n / 2), ws(n / 2);
    for (size_t k = 0; k < n / 2; ++k) {
        wc[k] = std::cos(NCO_2PI * (double)k / (double)n);
        ws[k] = -std::sin(NCO_2PI * (double)k / (double)n);
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const size_t half = len / 2, step = n / len;
        for (size_t s = 0; s < n; s += len)
            for (size_t k = 0; k < half; ++k) {
                const double c = wc[k * step], d = ws[k * step];
                const size_t p = s + k, q = p + half;
                const double tr = re[q] * c - im[q] * d, ti = re[q] * d + im[q] * c;
                re[q] = re[p] - tr; im[q] = im[p] - ti;
                re[p] += tr; im[p] += ti;
            }
    }
}

// rho = (N - P - 1) mod D in [0, D): N - P - 1 is -1 when P = N (L = 1), where C++'s % would give -1
inline long long fcfb_rho(long long N, long long P, long long D) { return ((N - P - 1) % D + D) % D; }

inline unsigned long long gcd_u(unsigned long long a, unsigned long long b) {
    while (b) { const unsigned long long t = a % b; a = b; b = t; }
    return a;
}

// G'[r] = DFT_N(g)[r] e^{sign 2 pi i r rho / N}, r < N, with g the rotated taps h[j] e^{+2 pi i (j inc mod 2^64) / 2^64}
// zero-padded to N; f64 throughout with the exact integer angle r rho mod N, rounded to f32 once.  The analysis bank
// takes sign = +1, the synthesis bank sign = -1.
inline void fc_spectrum(const float *h, long long L, uint64_t inc, long long N, long long rho, int sign, float2 *G) {
    std::vector<double> re((size_t)N, 0.0), im((size_t)N, 0.0);
    for (long long j = 0; j < L; ++j) {
        const double t = NCO_2PI * nco_turns((uint64_t)j * inc);
        re[j] = (double)h[j] * std::cos(t);
        im[j] = (double)h[j] * std::sin(t);
    }
    fft_f64(re, im);
    for (long long r = 0; r < N; ++r) {
        const long long q = (long long)(((unsigned long long)r * (unsigned long long)rho) % (unsigned long long)N);
        const double t = NCO_2PI * (double)q / (double)N, cs = std::cos(t), sn = (double)sign * std::sin(t);
        G[r] = make_float2((float)(re[r] * cs - im[r] * sn), (float)(re[r] * sn + im[r] * cs));
    }
}

}  // namespace sdr

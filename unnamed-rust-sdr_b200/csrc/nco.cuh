// nco.cuh -- the 64-bit NCO shared by the down-converter bank (ddc.cu), the fast-convolution bank (fcfb.cu) and the
// up-converter bank (duc.cu, which takes the conjugate of nco_rot): the exact derotation e^{-2 pi i phi / 2^64} on the
// device and the host-side f64 phase and rotated-taps helpers.
#pragma once
#include <cmath>
#include <vector>

#include "common.cuh"

namespace sdr {

// e^{-2 pi i phi / 2^64} from the exact 64-bit phase (phi read as signed: one turn = 2^64)
__device__ __forceinline__ float2 nco_rot(uint64_t phi) {
    double s, c;
    sincospi((double)(long long)phi * 0x1p-63, &s, &c);
    return make_float2((float)c, (float)-s);
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

}  // namespace sdr

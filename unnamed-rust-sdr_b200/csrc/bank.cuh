// bank.cuh -- device pieces shared by the per-channel resampler banks (rrb.cu, arb.cu): the flattened (channel, tile)
// grid and the carried frames of every channel.
#pragma once
#include <cuda_runtime.h>

namespace sdr {

// the channel whose tiles hold tile t: tile0[k] <= t < tile0[k + 1], k < C
__device__ __forceinline__ int bank_tile_channel(const long long *__restrict__ tile0, int C, long long t) {
    int a = 0, b = C;
    while (b - a > 1) {
        const int m = (a + b) >> 1;
        if (__ldg(tile0 + m) <= t) a = m;
        else b = m;
    }
    return a;
}

// the last H frames of (the H carried frames at hist_old + off, the call's row y of n frames) into hist_new + off, by
// the CTA's threads
__device__ __forceinline__ void bank_carry(const float2 *__restrict__ hist_old, const float2 *__restrict__ y,
                                           long long n, int H, long long off, float2 *__restrict__ hist_new) {
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        const long long s = n - H + j;
        hist_new[off + j] = s >= 0 ? __ldg(y + s) : __ldg(hist_old + off + H + s);
    }
}

}  // namespace sdr

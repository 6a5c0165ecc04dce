// arb_core.cuh -- the interpolant of the arbitrary-ratio resampler bank (K14), shared by arb.cu and tsync.cu so that
// both banks compute A(t) with the same device code: frame loads, and one fmaf chain per component over the channel's
// (h, d) table at the position's phase and 2^-24-truncated weight.
#pragma once
#include <cuda_runtime.h>

namespace sdr {

// frame j of a channel: hist[j] for j < 0 (hist points one past the carried frames), y[j] for 0 <= j < n, else 0
__device__ __forceinline__ float2 arb_load(const float2 *hist, const float2 *y, long long j, long long lo) {
    if (j < lo) return make_float2(0.f, 0.f);
    if (j < 0) return __ldg(hist + j);
    return __ldg(y + j);
}

// one term of a chain, in two steps: the interpolated tap c = fmaf(a, d, h) of table entry hd = (h, d), then c times
// frame v into acc
__device__ __forceinline__ float arb_tap(float2 hd, float a) { return __fmaf_rn(a, hd.y, hd.x); }
__device__ __forceinline__ void arb_acc(float c, float2 v, float2 &acc) {
    acc.x = __fmaf_rn(c, v.x, acc.x);
    acc.y = __fmaf_rn(c, v.y, acc.y);
}

// the chain of one output: T terms, frame n0 - i and table entry tb[i P] (tb = the table at ip).  CHECK = false when
// every frame read lies in the caller's row.
template <bool CHECK>
__device__ __forceinline__ float2 arb_chain(const float2 *__restrict__ tb, int T, int P, float a, const float2 *hist,
                                            const float2 *y, long long n0, long long lo) {
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll 4
    for (int i = 0; i < T; ++i) {
        const float2 hd = __ldg(tb + (long long)i * P);
        const float c = arb_tap(hd, a);
        const float2 v = CHECK ? arb_load(hist, y, n0 - i, lo) : __ldg(y + (n0 - i));
        arb_acc(c, v, acc);
    }
    return acc;
}

}  // namespace sdr

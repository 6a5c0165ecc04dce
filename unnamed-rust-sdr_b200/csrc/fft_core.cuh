// fft_core.cuh -- register-resident FFT building blocks shared by the FFT kernels (fft.cu) and the fused power-spectrum
// kernel (psd.cu): radix 2/4/8/16 butterflies and the 32-point DFT of the 1024-point warp kernel.
#pragma once
#include "common.cuh"

namespace sdr {

namespace {

constexpr float C_SQRT1_2 = 0.70710678118654752440f;
constexpr float C_COS_PI_8 = 0.92387953251128675613f;
constexpr float C_SIN_PI_8 = 0.38268343236508977173f;

__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }  // a * (-i)

// forward 4-point DFT in place on a, b, c, d -> X0..X3
template <bool PK = false>
__device__ __forceinline__ void dft4(float2 &a, float2 &b, float2 &c, float2 &d) {
    const float2 s02 = cadd_t<PK>(a, c), d02 = csub_t<PK>(a, c), s13 = cadd_t<PK>(b, d), d13 = mul_mi(csub_t<PK>(b, d));
    a = cadd_t<PK>(s02, s13);
    b = cadd_t<PK>(d02, d13);
    c = csub_t<PK>(s02, s13);
    d = csub_t<PK>(d02, d13);
}

// R-point forward DFT over v[0], v[S], ..., v[(R-1)S]; natural order in and out.
template <int R, int S, bool PK = false>
__device__ __forceinline__ void dft(float2 *v) {
    if (R == 2) {
        const float2 a = v[0], b = v[S];
        v[0] = cadd_t<PK>(a, b);
        v[S] = csub_t<PK>(a, b);
    } else if (R == 4) {
        dft4<PK>(v[0], v[S], v[2 * S], v[3 * S]);
    } else if (R == 8) {
        // n = c + 2a: U[c][r] = DFT4_a(v[c+2a]); X[r] = U0[r] + W8^r U1[r]; X[r+4] = U0[r] - W8^r U1[r]
        float2 e0 = v[0], e1 = v[2 * S], e2 = v[4 * S], e3 = v[6 * S];
        float2 o0 = v[S], o1 = v[3 * S], o2 = v[5 * S], o3 = v[7 * S];
        dft4<PK>(e0, e1, e2, e3);
        dft4<PK>(o0, o1, o2, o3);
        o1 = make_float2((o1.x + o1.y) * C_SQRT1_2, (o1.y - o1.x) * C_SQRT1_2);   // * W8^1 = (1-i)/sqrt2
        o2 = mul_mi(o2);                                                          // * W8^2 = -i
        o3 = make_float2((o3.y - o3.x) * C_SQRT1_2, -(o3.x + o3.y) * C_SQRT1_2);  // * W8^3 = (-1-i)/sqrt2
        v[0] = cadd_t<PK>(e0, o0); v[4 * S] = csub_t<PK>(e0, o0);
        v[S] = cadd_t<PK>(e1, o1); v[5 * S] = csub_t<PK>(e1, o1);
        v[2 * S] = cadd_t<PK>(e2, o2); v[6 * S] = csub_t<PK>(e2, o2);
        v[3 * S] = cadd_t<PK>(e3, o3); v[7 * S] = csub_t<PK>(e3, o3);
    } else {  // R == 16, S == 1
        // n = c + 4a: U[c][r] = DFT4_a(v[c+4a]); X[r+4q] = DFT4_c(W16^{c r} U[c][r])[q]
        float2 u[4][4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            u[c][0] = v[c * S]; u[c][1] = v[(c + 4) * S]; u[c][2] = v[(c + 8) * S]; u[c][3] = v[(c + 12) * S];
            dft4<PK>(u[c][0], u[c][1], u[c][2], u[c][3]);
        }
        const float2 w1 = make_float2(C_COS_PI_8, -C_SIN_PI_8);
        const float2 w2 = make_float2(C_SQRT1_2, -C_SQRT1_2);
        const float2 w3 = make_float2(C_SIN_PI_8, -C_COS_PI_8);
        const float2 w6 = make_float2(-C_SQRT1_2, -C_SQRT1_2);
        const float2 w9 = make_float2(-C_COS_PI_8, C_SIN_PI_8);
        u[1][1] = cmul(u[1][1], w1); u[1][2] = cmul(u[1][2], w2); u[1][3] = cmul(u[1][3], w3);
        u[2][1] = cmul(u[2][1], w2); u[2][2] = mul_mi(u[2][2]);   u[2][3] = cmul(u[2][3], w6);
        u[3][1] = cmul(u[3][1], w3); u[3][2] = cmul(u[3][2], w6); u[3][3] = cmul(u[3][3], w9);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            dft4<PK>(u[0][r], u[1][r], u[2][r], u[3][r]);
            v[r * S] = u[0][r]; v[(r + 4) * S] = u[1][r]; v[(r + 8) * S] = u[2][r]; v[(r + 12) * S] = u[3][r];
        }
    }
}

// cos / sin of pi*r/16, r = 0..8 (first quadrant); W32^r = (cos, -sin) extended by symmetry
__host__ __device__ constexpr float w32_q(int r) {
    return r == 0 ? 1.0f : r == 1 ? 0.98078528040323044913f : r == 2 ? 0.92387953251128675613f
         : r == 3 ? 0.83146961230254523708f : r == 4 ? 0.70710678118654752440f : r == 5 ? 0.55557023301960222474f
         : r == 6 ? 0.38268343236508977173f : r == 7 ? 0.19509032201612826785f : 0.0f;
}
__host__ __device__ constexpr float w32_cos(int r) { return r <= 8 ? w32_q(r) : -w32_q(16 - r); }
__host__ __device__ constexpr float w32_sin(int r) { return r <= 8 ? w32_q(8 - r) : w32_q(r - 8); }

// 32-point forward DFT, v (natural order) -> w (natural order).  n = c + 2a: two 16-point DFTs over the even
// and odd inputs, then X[r] = U0[r] + W32^r U1[r], X[r+16] = U0[r] - W32^r U1[r].
template <bool PK = false>
__device__ __forceinline__ void dft32(float2 (&v)[32], float2 (&w)[32]) {
    dft<16, 2, PK>(v);
    dft<16, 2, PK>(v + 1);
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const float2 u0 = v[2 * r], u1 = v[2 * r + 1];
        float2 t;
        if (r == 0) t = u1;
        else if (r == 8) t = mul_mi(u1);
        else if (r == 4) t = make_float2((u1.x + u1.y) * C_SQRT1_2, (u1.y - u1.x) * C_SQRT1_2);
        else if (r == 12) t = make_float2((u1.y - u1.x) * C_SQRT1_2, -(u1.x + u1.y) * C_SQRT1_2);
        else t = cmul(u1, make_float2(w32_cos(r), -w32_sin(r)));
        w[r] = cadd_t<PK>(u0, t);
        w[r + 16] = csub_t<PK>(u0, t);
    }
}

}  // namespace

}  // namespace sdr

// psd_mirror_test.cpp -- averaged power spectra through the C++ host mirror (host/sdr.hpp): fft::PowerSpectra against
// the crate's own chain run through the same mirror -- fft::WindowSpectra (window -> decimate -> fft::fft), |.|^2 and
// the mean of K in f64; streaming, clone and reset give the same bits as one call.
// Built and run by tests/test_gpu_psd.py (needs a GPU: there is no CPU fallback).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../unnamed-rust-sdr_b200/host/sdr.hpp"

using namespace sdr;

static int fails = 0;
#define EXPECT(cond, ...)                               \
    do {                                                \
        if (!(cond)) {                                  \
            ++fails;                                    \
            printf("FAIL %s:%d: ", __FILE__, __LINE__); \
            printf(__VA_ARGS__);                        \
            printf("\n");                               \
        }                                               \
    } while (0)

static uint64_t splitmix(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

static bool same_bits(const std::vector<float> &a, const std::vector<float> &b) {
    return a.size() == b.size() && std::memcmp(a.data(), b.data(), a.size() * sizeof(float)) == 0;
}

int main() {
    const size_t n = 300000, H = 512, K = 40;
    const float rate = 1024000.0f;
    std::vector<uint8_t> raw(2 * n);
    for (size_t i = 0; i < 2 * n; ++i) raw[i] = (uint8_t)(splitmix(i ^ 0x9D5B200) >> 56);

    for (size_t N : {(size_t)1024, (size_t)1000}) {
        // the composition: WindowSpectra(duration = N / rate, fps = rate / H) then |.|^2 and the mean of K
        fft::WindowSpectra ws(rate, (float)N / rate, rate / (float)H, true);
        EXPECT(ws.window() == N, "window %zu", ws.window());
        std::vector<Complex> X;
        const size_t nw = ws.process(raw.data(), n, X);
        const size_t G = nw / K;
        fft::PowerSpectra ps(N, H, K, {}, true);
        std::vector<float> P;
        EXPECT(ps.process(raw.data(), n, P) == G && G == (n / H) / K, "spectra %zu", G);
        EXPECT(ps.last_path() == (N == 1024 ? 2 : 1), "path %d", ps.last_path());
        const double bar = 2e-5 * std::log2((double)N);
        for (size_t g = 0; g < G; ++g) {
            std::vector<double> want(N, 0.0);
            double mx = 0, err = 0;
            for (size_t j = g * K; j < (g + 1) * K; ++j)
                for (size_t k = 0; k < N; ++k) want[k] += std::norm(std::complex<double>(X[j * N + k])) / K;
            for (size_t k = 0; k < N; ++k) mx = std::max(mx, want[k]);
            for (size_t k = 0; k < N; ++k) err = std::max(err, std::fabs(P[g * N + k] - want[k]));
            EXPECT(err <= bar * mx, "N %zu spectrum %zu err %g max %g", N, g, err, mx);
        }
        // streaming in ragged blocks, a clone taken mid-group, reset
        fft::PowerSpectra st(N, H, K, {}, true);
        std::vector<float> Q, R;
        size_t at = 0, step = 1;
        while (at < n / 2) {
            const size_t m = std::min(step, n / 2 - at);
            st.process(raw.data() + 2 * at, m, Q);
            at += m;
            step = step * 3 + 7;
        }
        fft::PowerSpectra cl(st);
        R = Q;
        st.process(raw.data() + 2 * at, n - at, Q);
        cl.process(raw.data() + 2 * at, n - at, R);
        EXPECT(same_bits(Q, P), "N %zu blocks != one call", N);
        EXPECT(same_bits(R, P), "N %zu clone != one call", N);
        st.reset();
        std::vector<float> S;
        st.process(raw.data(), n, S);
        EXPECT(same_bits(S, P), "N %zu reset != one call", N);
    }
    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("PSD MIRROR OK\n");
    return 0;
}

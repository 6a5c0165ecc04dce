// pfb_mirror_test.cpp -- the polyphase filter bank through the C++ host mirror (host/sdr.hpp): every channel of
// filter::Pfb against the crate's own composition, filter::Fir<Complex, Complex>(h[n] e^{+2 pi i k n / M}) with
// Decimate(D), run through the same mirror; streaming, clone and u8 input.
// Built and run by tests/test_gpu_pfb.py (needs a GPU: there is no CPU fallback).
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

static std::vector<float> lowpass(int n, double fc) {  // fc in cycles per sample
    std::vector<double> h(n);
    double sum = 0;
    for (int k = 0; k < n; ++k) {
        double t = k - (n - 1) / 2.0, a = 2 * fc;
        double s = (t == 0) ? 1.0 : std::sin(M_PI * a * t) / (M_PI * a * t);
        h[k] = a * s * (0.54 - 0.46 * std::cos(2 * M_PI * k / (n - 1)));
        sum += h[k];
    }
    std::vector<float> o(n);
    for (int k = 0; k < n; ++k) o[k] = (float)(h[k] / sum);
    return o;
}

static bool same_bits(const std::vector<Complex> &a, const std::vector<Complex> &b) {
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i)
        if (std::memcmp(&a[i], &b[i], sizeof(Complex)) != 0) return false;
    return true;
}

int main() {
    const size_t M = 16, D = 12, n = 6000;
    const std::vector<float> h = lowpass(5 * (int)M + 3, 0.5 / M);
    std::vector<uint8_t> raw(2 * n);
    for (size_t i = 0; i < 2 * n; ++i) raw[i] = (uint8_t)(splitmix(i ^ 0x5D12B200) >> 56);
    std::vector<Complex> x(n);
    for (size_t i = 0; i < n; ++i) x[i] = Complex((raw[2 * i] - 128.0f) / 128.0f, (raw[2 * i + 1] - 128.0f) / 128.0f);

    // ---- every channel against Fir<Complex, Complex>(g_k) + Decimate(D) ----
    filter::Pfb bank(h, M, D);
    std::vector<Complex> y;
    const size_t nf = bank.process(x.data(), n, y);
    EXPECT(nf == n / D && y.size() == nf * M, "frames %zu", nf);
    double peak = 0, err = 0;
    for (size_t k = 0; k < M; ++k) {
        std::vector<Complex> g(h.size());
        for (size_t i = 0; i < h.size(); ++i) {
            const double a = 2 * M_PI * (double)((k * i) % M) / (double)M;
            g[i] = Complex((float)(h[i] * std::cos(a)), (float)(h[i] * std::sin(a)));
        }
        filter::Fir<Complex, Complex> fir(g, D);
        std::vector<Complex> ref;
        fir.process(x.data(), n, ref);
        EXPECT(ref.size() == nf, "channel %zu: %zu outputs", k, ref.size());
        for (size_t m = 0; m < nf && m < ref.size(); ++m) {
            peak = std::max(peak, (double)std::abs(ref[m]));
            err = std::max(err, (double)std::abs(ref[m] - y[m * M + k]));
        }
    }
    EXPECT(err <= 1e-5 * std::log2((double)M) * peak, "max |pfb - fir| = %g of peak %g", err, peak);

    // ---- ragged blocks, clone mid-stream, u8 input: the same bits ----
    filter::Pfb s(h, M, D);
    std::vector<Complex> part, cat;
    size_t pos = 0;
    for (size_t blk : {1ul, 7ul, 0ul, 1000ul}) {
        s.process(x.data() + pos, blk, part);
        cat.insert(cat.end(), part.begin(), part.end());
        pos += blk;
    }
    filter::Pfb c(s);
    std::vector<Complex> rest_s, rest_c;
    s.process(x.data() + pos, n - pos, rest_s);
    c.process(x.data() + pos, n - pos, rest_c);
    EXPECT(same_bits(rest_s, rest_c), "clone diverged");
    cat.insert(cat.end(), rest_s.begin(), rest_s.end());
    EXPECT(same_bits(cat, y), "blocked stream differs from one call");
    filter::Pfb u8(h, M, D, true);
    std::vector<Complex> yu;
    u8.process(raw.data(), n, yu);
    EXPECT(same_bits(yu, y), "u8 input differs from its unpacked c64");
    s.reset();
    std::vector<Complex> again;
    s.process(x.data(), n, again);
    EXPECT(same_bits(again, y), "reset differs from a fresh handle");

    // ---- channel-major is the transpose ----
    filter::Pfb cm(h, M, D, false, SDR_PFB_CHANNEL_MAJOR);
    std::vector<Complex> yt;
    cm.process(x.data(), n, yt);
    bool tr = yt.size() == y.size();
    for (size_t m = 0; tr && m < nf; ++m)
        for (size_t k = 0; k < M; ++k) tr = tr && std::memcmp(&yt[k * nf + m], &y[m * M + k], sizeof(Complex)) == 0;
    EXPECT(tr, "channel-major is not the transpose");

    if (fails) return 1;
    printf("PFB MIRROR OK (M=%zu D=%zu L=%zu, %zu frames, max err %.3g of %.3g)\n", M, D, h.size(), nf, err, peak);
    return 0;
}

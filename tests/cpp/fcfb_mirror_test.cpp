// fcfb_mirror_test.cpp -- the fast-convolution channel bank through the C++ host mirror (host/sdr.hpp): every channel
// of filter::Fcfb against the crate's own composition run through the same mirror -- the stream mixed down by a 64-bit
// NCO (what a caller writes with Signal::map), filter::Fir(h) with Decimate(D_k); streaming, clone and reset.
// Built and run by tests/test_gpu_fcfb.py (needs a GPU: there is no CPU fallback).
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
    const size_t C = 3, n = 20000, L = 127;
    const double rate = 2.4e6;
    const std::vector<double> freqs = {312.5e3, -687e3, 100e3};
    const std::vector<size_t> D = {8, 10, 1};
    const std::vector<float> h = lowpass((int)L, 100e3 / rate);
    std::vector<uint8_t> raw(2 * n);
    for (size_t i = 0; i < 2 * n; ++i) raw[i] = (uint8_t)(splitmix(i ^ 0x5D12B200) >> 56);
    std::vector<Complex> x(n);
    for (size_t i = 0; i < n; ++i) x[i] = Complex((raw[2 * i] - 128.0f) / 128.0f, (raw[2 * i + 1] - 128.0f) / 128.0f);

    // ---- every channel against a mixer (Signal::map over a 64-bit NCO) + Fir(h) + Decimate(D_k) ----
    filter::Fcfb bank(h, L, freqs, rate, D);
    std::vector<std::vector<Complex>> y;
    bank.process(raw.data(), n, y);
    EXPECT(y.size() == C, "channels %zu", y.size());
    double worst = 0;
    for (size_t k = 0; k < C && k < y.size(); ++k) {
        EXPECT(y[k].size() <= n / D[k] && y[k].size() + 4096 / D[k] >= n / D[k], "channel %zu: %zu outputs", k,
               y[k].size());
        const uint64_t inc = sdr_ddc_phase_increment(freqs[k], rate);
        std::vector<Complex> z(n);
        for (size_t i = 0; i < n; ++i) {
            const double t = -2 * M_PI * (double)(int64_t)((uint64_t)i * inc) * 0x1p-64;
            z[i] = x[i] * Complex((float)std::cos(t), (float)std::sin(t));
        }
        std::vector<Complex> g(h.begin(), h.end());
        filter::Fir<Complex, Complex> fir(g, D[k]);
        std::vector<Complex> ref;
        fir.process(z.data(), n, ref);
        double peak = 0, err = 0;
        for (size_t m = 0; m < ref.size(); ++m) peak = std::max(peak, (double)std::abs(ref[m]));
        for (size_t m = 0; m < y[k].size() && m < ref.size(); ++m) err = std::max(err, (double)std::abs(ref[m] - y[k][m]));
        // the bank's bar 2e-5 log2(N) plus the composition's own f32 error
        EXPECT(err <= (2e-5 * 10 + 1e-5) * peak, "channel %zu: max |fcfb - mix+fir| = %g of peak %g", k, err, peak);
        worst = std::max(worst, err / peak);
    }

    // ---- ragged blocks (1-sample calls, calls ending mid-block), clone mid-stream, reset: the same bits ----
    filter::Fcfb s(h, L, freqs, rate, D);
    std::vector<std::vector<Complex>> part, rows(C);
    size_t pos = 0;
    auto append = [&](const std::vector<std::vector<Complex>> &p) {
        for (size_t k = 0; k < C; ++k) rows[k].insert(rows[k].end(), p[k].begin(), p[k].end());
    };
    for (size_t blk : {1ul, 7ul, 0ul, 1000ul, 4099ul, 1ul}) {
        s.process(raw.data() + 2 * pos, blk, part);
        append(part);
        pos += blk;
    }
    filter::Fcfb c(s);
    std::vector<std::vector<Complex>> rest_s, rest_c;
    s.process(raw.data() + 2 * pos, n - pos, rest_s);
    c.process(raw.data() + 2 * pos, n - pos, rest_c);
    bool same = true;
    for (size_t k = 0; k < C; ++k) same = same && same_bits(rest_s[k], rest_c[k]);
    EXPECT(same, "clone diverged");
    append(rest_s);
    same = true;
    for (size_t k = 0; k < C; ++k) same = same && same_bits(rows[k], y[k]);
    EXPECT(same, "blocked stream differs from one call");
    s.reset();
    std::vector<std::vector<Complex>> again;
    s.process(raw.data(), n, again);
    same = true;
    for (size_t k = 0; k < C; ++k) same = same && same_bits(again[k], y[k]);
    EXPECT(same, "reset differs from a fresh handle");

    if (fails) return 1;
    printf("FCFB MIRROR OK (C=%zu D={8,10,1} L=%zu, max err %.3g of peak)\n", C, L, worst);
    return 0;
}

// rrb_mirror_test.cpp -- the rational resampler bank through the C++ host mirror (host/sdr.hpp): filter::Rrb against
// the crate's own composition, each channel zero-stuffed by I_k, run through filter::Fir<float, Complex>(h) of the same
// mirror and decimated by D_k; ragged calls with a different split per channel, clone and reset give the bits of one
// call.  Built and run by tests/test_gpu_rrb.py (needs a GPU: there is no CPU fallback).
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

static std::vector<float> lowpass(int n, double fc, double gain) {  // fc in cycles per sample
    std::vector<double> h(n);
    double sum = 0;
    for (int k = 0; k < n; ++k) {
        double t = k - (n - 1) / 2.0, a = 2 * fc;
        double s = (t == 0) ? 1.0 : std::sin(M_PI * a * t) / (M_PI * a * t);
        h[k] = a * s * (0.54 - 0.46 * std::cos(2 * M_PI * k / (n - 1)));
        sum += h[k];
    }
    std::vector<float> o(n);
    for (int k = 0; k < n; ++k) o[k] = (float)(gain * h[k] / sum);
    return o;
}

static bool same_bits(const std::vector<Complex> &a, const std::vector<Complex> &b) {
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i)
        if (std::memcmp(&a[i], &b[i], sizeof(Complex)) != 0) return false;
    return true;
}

int main() {
    const std::vector<size_t> I = {4, 147, 75}, D = {25, 160, 64};
    const size_t C = I.size(), L = 441, nf = 3000;
    const std::vector<float> h = lowpass((int)L, 0.4 / 160, 1.0);
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i ^ 0x44B200ull);
        y[i] = Complex((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f, (float)((r >> 8) & 0xFFFF) / 32768.0f - 1.0f);
    }

    // ---- against zero-stuff + Fir<float, Complex>(h) + keep (r+1) D - 1 ----
    filter::Rrb bank(h, L, I, D);
    std::vector<std::vector<Complex>> z;
    bank.process(y.data(), std::vector<size_t>(C, nf), nf, z);
    double worst = 0;
    for (size_t k = 0; k < C; ++k) {
        std::vector<Complex> s(nf * I[k], Complex(0, 0)), u;
        for (size_t m = 0; m < nf; ++m) s[(m + 1) * I[k] - 1] = y[k * nf + m];
        filter::Fir<float, Complex> fir(h);
        fir.process(s.data(), s.size(), u);
        const size_t want = nf * I[k] / D[k];
        EXPECT(z[k].size() == want, "channel %zu: %zu outputs, want %zu", k, z[k].size(), want);
        double peak = 0, err = 0;
        for (size_t r = 0; r < z[k].size() && (r + 1) * D[k] - 1 < u.size(); ++r) {
            const Complex ref = u[(r + 1) * D[k] - 1];
            peak = std::max(peak, (double)std::abs(ref));
            err = std::max(err, (double)std::abs(ref - z[k][r]));
        }
        EXPECT(err <= 1e-5 * peak, "channel %zu: max |rrb - fir decimate| = %g of peak %g", k, err, peak);
        worst = std::max(worst, err / peak);
    }

    // ---- ragged calls, a different split per channel, clone mid-stream, reset: the same bits ----
    filter::Rrb s(h, L, I, D);
    std::vector<std::vector<Complex>> cat(C), part;
    std::vector<size_t> pos(C, 0);
    const size_t splits[4][3] = {{1, 7, 0}, {100, 3, 55}, {0, 250, 9}, {640, 1, 333}};
    for (const auto &sp : splits) {
        std::vector<Complex> rows(C * nf, Complex(0, 0));
        std::vector<size_t> n(C);
        for (size_t k = 0; k < C; ++k) {
            n[k] = sp[k];
            std::copy(y.begin() + k * nf + pos[k], y.begin() + k * nf + pos[k] + n[k], rows.begin() + k * nf);
            pos[k] += n[k];
        }
        s.process(rows.data(), n, nf, part);
        for (size_t k = 0; k < C; ++k) cat[k].insert(cat[k].end(), part[k].begin(), part[k].end());
    }
    filter::Rrb c(s);
    std::vector<Complex> rest(C * nf, Complex(0, 0));
    std::vector<size_t> n(C);
    for (size_t k = 0; k < C; ++k) {
        n[k] = nf - pos[k];
        std::copy(y.begin() + k * nf + pos[k], y.begin() + (k + 1) * nf, rest.begin() + k * nf);
    }
    std::vector<std::vector<Complex>> rs, rc;
    s.process(rest.data(), n, nf, rs);
    c.process(rest.data(), n, nf, rc);
    for (size_t k = 0; k < C; ++k) {
        EXPECT(same_bits(rs[k], rc[k]), "channel %zu: clone diverged", k);
        cat[k].insert(cat[k].end(), rs[k].begin(), rs[k].end());
        EXPECT(same_bits(cat[k], z[k]), "channel %zu: blocked stream differs from one call", k);
    }
    s.reset();
    std::vector<std::vector<Complex>> again;
    s.process(y.data(), std::vector<size_t>(C, nf), nf, again);
    for (size_t k = 0; k < C; ++k) EXPECT(same_bits(again[k], z[k]), "channel %zu: reset differs", k);

    if (fails) return 1;
    printf("RRB MIRROR OK (C=%zu L=%zu, ratios 4/25 147/160 75/64, max err %.3g of peak)\n", C, L, worst);
    return 0;
}

// duc_mirror_test.cpp -- the up-converter bank through the C++ host mirror (host/sdr.hpp): filter::Duc against the
// crate's own composition, each channel zero-stuffed by I, run through filter::Fir<float, Complex>(h_k) of the same
// mirror, mixed up by the exact 64-bit NCO phase and summed; streaming with a row stride, clone, reset, and the
// Ddc -> Duc round trip.  Built and run by tests/test_gpu_duc.py (needs a GPU: there is no CPU fallback).
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
    const size_t C = 3, I = 8, L = 127, nf = 500;
    const uint64_t F = (1ull << 40) + 12345;
    const std::vector<double> freqs = {-0.3, 0.05, 0.27};
    const std::vector<float> h = lowpass((int)L, 0.5 / I, (double)I);
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i ^ 0xD0C5B200ull);
        y[i] = Complex((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f, (float)((r >> 8) & 0xFFFF) / 32768.0f - 1.0f);
    }

    // ---- against zero-stuff + Fir<float, Complex>(h) + NCO mix + sum ----
    filter::Duc bank(h, L, freqs, 1.0, I, F);
    std::vector<Complex> x;
    const size_t n = bank.process(y.data(), nf, nf, x);
    EXPECT(n == nf * I && x.size() == n, "outputs %zu", n);
    std::vector<std::complex<double>> ref(nf * I, 0.0);
    for (size_t k = 0; k < C; ++k) {
        const uint64_t inc = sdr_ddc_phase_increment(freqs[k], 1.0);
        std::vector<Complex> z(nf * I, Complex(0, 0)), o;
        for (size_t m = 0; m < nf; ++m) z[(m + 1) * I - 1] = y[k * nf + m];
        filter::Fir<float, Complex> fir(h);
        fir.process(z.data(), z.size(), o);
        EXPECT(o.size() == nf * I, "channel %zu: %zu outputs", k, o.size());
        for (size_t t = 0; t < o.size() && t < ref.size(); ++t) {
            const double a = 2 * M_PI * (double)(int64_t)((F + t) * inc) * 0x1p-64;
            ref[t] += std::complex<double>(o[t].real(), o[t].imag()) * std::complex<double>(std::cos(a), std::sin(a));
        }
    }
    double peak = 0, err = 0;
    for (size_t t = 0; t < n; ++t) {
        peak = std::max(peak, std::abs(ref[t]));
        err = std::max(err, std::abs(ref[t] - std::complex<double>(x[t].real(), x[t].imag())));
    }
    EXPECT(err <= 1e-5 * peak, "max |duc - fir mix sum| = %g of peak %g", err, peak);

    // ---- ragged calls on rows of a wider buffer, clone mid-stream, reset: the same bits ----
    filter::Duc s(h, L, freqs, 1.0, I, F);
    std::vector<Complex> part, cat;
    size_t pos = 0;
    for (size_t blk : {1ul, 7ul, 0ul, 100ul}) {
        s.process(y.data() + pos, blk, nf, part);
        cat.insert(cat.end(), part.begin(), part.end());
        pos += blk;
    }
    filter::Duc c(s);
    std::vector<Complex> rest_s, rest_c;
    s.process(y.data() + pos, nf - pos, nf, rest_s);
    c.process(y.data() + pos, nf - pos, nf, rest_c);
    EXPECT(same_bits(rest_s, rest_c), "clone diverged");
    cat.insert(cat.end(), rest_s.begin(), rest_s.end());
    EXPECT(same_bits(cat, x), "blocked stream differs from one call");
    s.reset();
    std::vector<Complex> again;
    s.process(y.data(), nf, nf, again);
    EXPECT(same_bits(again, x), "reset differs from a fresh handle");

    // ---- Ddc -> Duc: three tones at the channel centres come back delayed by L - 1 (Hamming pair) ----
    const size_t ns = 400 * I;
    std::vector<Complex> in(ns, Complex(0, 0));
    for (size_t k = 0; k < C; ++k) {
        const uint64_t inc = sdr_ddc_phase_increment(freqs[k], 1.0);
        for (size_t t = 0; t < ns; ++t) {
            const double a = 2 * M_PI * (double)(int64_t)((F + t) * inc) * 0x1p-64;
            in[t] += Complex((float)(0.3 * std::cos(a)), (float)(0.3 * std::sin(a)));
        }
    }
    const std::vector<float> ha = lowpass((int)L, 0.5 / I, 1.0);
    filter::Ddc ana(ha, L, freqs, 1.0, I, false, F);
    std::vector<Complex> rows, back;
    const size_t fn = ana.process(in.data(), ns, rows);
    const size_t d = L - 1;
    filter::Duc syn(h, L, freqs, 1.0, I, F - d);
    syn.process(rows.data(), fn, fn, back);
    double pe = 0, pw = 0;
    for (size_t t = 2 * d; t < back.size(); ++t) {
        pw += std::norm(in[t - d]);
        pe += std::norm(back[t] - in[t - d]);
    }
    const double snr = 10 * std::log10(pw / pe);
    EXPECT(back.size() == ns && snr > 40, "round trip: %zu samples, %.1f dB", back.size(), snr);

    if (fails) return 1;
    printf("DUC MIRROR OK (C=%zu I=%zu L=%zu, %zu outputs, max err %.3g of %.3g, round trip %.1f dB)\n", C, I, L, n,
           err, peak, snr);
    return 0;
}

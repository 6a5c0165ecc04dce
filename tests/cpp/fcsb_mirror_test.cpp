// fcsb_mirror_test.cpp -- the fast-convolution synthesis bank through the C++ host mirror (host/sdr.hpp): the sum of
// filter::Fcsb's channels against the crate's own composition run through the same mirror -- each channel zero-stuffed
// by its own I_k, filter::Fir<f32, Complex>(h), mixed up by a 64-bit NCO (Signal::map) and summed; streaming, clone
// and reset; the Fcfb -> Fcsb round trip at mixed rates.  Built and run by tests/test_gpu_fcsb.py (needs a GPU: there
// is no CPU fallback).
#include <cmath>
#include <complex>
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
    const size_t C = 3, L = 127, Il = 40, n = 100 * Il;
    const uint64_t F = (1ull << 40) + 12345;
    const std::vector<double> freqs = {-0.3, 0.05, 0.27};
    const std::vector<size_t> I = {8, 10, 40};
    std::vector<float> h;  // one row per channel, gain I_k
    for (size_t k = 0; k < C; ++k) {
        const std::vector<float> r = lowpass((int)L, 0.5 / I[k], (double)I[k]);
        h.insert(h.end(), r.begin(), r.end());
    }
    const size_t stride = n / 8;
    std::vector<Complex> y(C * stride, Complex(0, 0));
    for (size_t k = 0; k < C; ++k)
        for (size_t m = 0; m < n / I[k]; ++m) {
            const uint64_t r = splitmix((k * stride + m) ^ 0xFC5BB200ull);
            y[k * stride + m] = Complex((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f,
                                        (float)((r >> 8) & 0xFFFF) / 32768.0f - 1.0f);
        }

    // ---- against zero-stuff + Fir<float, Complex>(h_k) + NCO mix + sum ----
    filter::Fcsb bank(h, L, freqs, 1.0, I, F);
    std::vector<Complex> x;
    const size_t got = bank.process(y.data(), n, stride, x);
    EXPECT(got <= n && got + 4096 >= n && x.size() == got, "outputs %zu", got);
    std::vector<std::complex<double>> ref(n, 0.0);
    for (size_t k = 0; k < C; ++k) {
        const uint64_t inc = sdr_ddc_phase_increment(freqs[k], 1.0);
        std::vector<Complex> z(n, Complex(0, 0)), o;
        for (size_t m = 0; m < n / I[k]; ++m) z[(m + 1) * I[k] - 1] = y[k * stride + m];
        std::vector<float> hk(h.begin() + k * L, h.begin() + (k + 1) * L);
        filter::Fir<float, Complex> fir(hk);
        fir.process(z.data(), z.size(), o);
        for (size_t t = 0; t < o.size() && t < ref.size(); ++t) {
            const double a = 2 * M_PI * (double)(int64_t)((F + t) * inc) * 0x1p-64;
            ref[t] += std::complex<double>(o[t].real(), o[t].imag()) * std::complex<double>(std::cos(a), std::sin(a));
        }
    }
    double peak = 0, err = 0;
    for (size_t t = 0; t < got; ++t) {
        peak = std::max(peak, std::abs(ref[t]));
        err = std::max(err, std::abs(ref[t] - std::complex<double>(x[t].real(), x[t].imag())));
    }
    // the bank's bar 2e-5 log2(N) plus the composition's own f32 error
    EXPECT(err <= (2e-5 * 10 + 1e-5) * peak, "max |fcsb - fir mix sum| = %g of peak %g", err, peak);

    // ---- ragged calls (one Il, mid-block ends), clone mid-stream, reset: the same bits ----
    filter::Fcsb s(h, L, freqs, 1.0, I, F);
    std::vector<Complex> part, cat;
    size_t pos = 0;
    for (size_t blk : {1ul, 7ul, 0ul, 30ul, 1ul}) {
        std::vector<Complex> sub(C * stride);
        for (size_t k = 0; k < C; ++k)
            std::memcpy(&sub[k * stride], &y[k * stride + pos / I[k]], blk * Il / I[k] * sizeof(Complex));
        s.process(sub.data(), blk * Il, stride, part);
        cat.insert(cat.end(), part.begin(), part.end());
        pos += blk * Il;
    }
    filter::Fcsb c(s);
    std::vector<Complex> rest(C * stride), rest_s, rest_c;
    for (size_t k = 0; k < C; ++k)
        std::memcpy(&rest[k * stride], &y[k * stride + pos / I[k]], (n - pos) / I[k] * sizeof(Complex));
    s.process(rest.data(), n - pos, stride, rest_s);
    c.process(rest.data(), n - pos, stride, rest_c);
    EXPECT(same_bits(rest_s, rest_c), "clone diverged");
    cat.insert(cat.end(), rest_s.begin(), rest_s.end());
    EXPECT(same_bits(cat, x), "blocked stream differs from one call");
    s.reset();
    std::vector<Complex> again;
    s.process(y.data(), n, stride, again);
    EXPECT(same_bits(again, x), "reset differs from a fresh handle");

    // ---- Fcfb -> Fcsb: tones at the channel centres come back delayed by Lr - 1 (Hamming pairs, D_k = I_k; long
    // enough that the images of I = 40 fall in the stop band) ----
    const size_t ns = 200 * Il, Lr = 511;
    std::vector<Complex> in(ns + 8192, Complex(0, 0));
    for (size_t k = 0; k < C; ++k) {
        const uint64_t inc = sdr_ddc_phase_increment(freqs[k], 1.0);
        for (size_t t = 0; t < ns; ++t) {
            const double a = 2 * M_PI * (double)(int64_t)((F + t) * inc) * 0x1p-64;
            in[t] += Complex((float)(0.3 * std::cos(a)), (float)(0.3 * std::sin(a)));
        }
    }
    std::vector<float> ha, hs;
    for (size_t k = 0; k < C; ++k) {
        const std::vector<float> a = lowpass((int)Lr, 0.5 / I[k], 1.0), b = lowpass((int)Lr, 0.5 / I[k], (double)I[k]);
        ha.insert(ha.end(), a.begin(), a.end());
        hs.insert(hs.end(), b.begin(), b.end());
    }
    filter::Fcfb ana(ha, Lr, freqs, 1.0, I, false, F);
    std::vector<std::vector<Complex>> rows;
    ana.process(in.data(), in.size(), rows);  // the stream and a drain of zeros
    const size_t nt = rows[0].size() * I[0], rs = rows[0].size();
    std::vector<Complex> packed(C * rs, Complex(0, 0)), back;
    for (size_t k = 0; k < C; ++k) {
        EXPECT(rows[k].size() * I[k] == nt, "channel %zu: %zu rows", k, rows[k].size());
        std::copy(rows[k].begin(), rows[k].end(), packed.begin() + k * rs);
    }
    const size_t d = Lr - 1;
    filter::Fcsb syn(hs, Lr, freqs, 1.0, I, F - d);
    syn.process(packed.data(), nt, rs, back);
    double pe = 0, pw = 0;
    for (size_t t = 2 * d; t < ns && t < back.size(); ++t) {
        pw += std::norm(in[t - d]);
        pe += std::norm(back[t] - in[t - d]);
    }
    const double snr = 10 * std::log10(pw / pe);
    EXPECT(back.size() >= ns && snr > 40, "round trip: %zu samples, %.1f dB", back.size(), snr);

    if (fails) return 1;
    printf("FCSB MIRROR OK (C=%zu I={8,10,40} L=%zu, %zu outputs, max err %.3g of %.3g, round trip %.1f dB)\n", C, L,
           got, err, peak, snr);
    return 0;
}

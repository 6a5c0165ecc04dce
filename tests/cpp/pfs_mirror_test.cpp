// pfs_mirror_test.cpp -- the polyphase synthesis bank through the C++ host mirror (host/sdr.hpp): filter::Pfs against
// the crate's own composition, each channel zero-stuffed by D and run through filter::Fir<Complex, Complex>(f[n]
// e^{+2 pi i k n / M}) of the same mirror, summed; streaming, clone, reset, channel-major input and the
// Pfb -> Pfs round trip.  Built and run by tests/test_gpu_pfs.py (needs a GPU: there is no CPU fallback).
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
    const size_t M = 16, D = 8, nf = 400;
    const std::vector<float> f = lowpass(6 * (int)M + 5, 1.0 / M, (double)D);
    std::vector<Complex> y(nf * M);
    for (size_t i = 0; i < nf * M; ++i) {
        const uint64_t r = splitmix(i ^ 0x5F5B200ull);
        y[i] = Complex((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f, (float)((r >> 8) & 0xFFFF) / 32768.0f - 1.0f);
    }

    // ---- against zero-stuff + Fir<Complex, Complex>(f_k) + sum ----
    filter::Pfs bank(f, M, D);
    std::vector<Complex> x;
    const size_t n = bank.process(y.data(), nf, x);
    EXPECT(n == nf * D && x.size() == n, "outputs %zu", n);
    std::vector<Complex> ref(nf * D, Complex(0, 0));
    for (size_t k = 0; k < M; ++k) {
        std::vector<Complex> g(f.size());
        for (size_t i = 0; i < f.size(); ++i) {
            const double a = 2 * M_PI * (double)((k * i) % M) / (double)M;
            g[i] = Complex((float)(f[i] * std::cos(a)), (float)(f[i] * std::sin(a)));
        }
        std::vector<Complex> z(nf * D, Complex(0, 0)), o;
        for (size_t m = 0; m < nf; ++m) z[(m + 1) * D - 1] = y[m * M + k];
        filter::Fir<Complex, Complex> fir(g);
        fir.process(z.data(), z.size(), o);
        EXPECT(o.size() == nf * D, "channel %zu: %zu outputs", k, o.size());
        for (size_t t = 0; t < o.size() && t < ref.size(); ++t) ref[t] += o[t];
    }
    double peak = 0, err = 0;
    for (size_t t = 0; t < n; ++t) {
        peak = std::max(peak, (double)std::abs(ref[t]));
        err = std::max(err, (double)std::abs(ref[t] - x[t]));
    }
    EXPECT(err <= 1e-5 * std::log2((double)M) * peak, "max |pfs - fir sum| = %g of peak %g", err, peak);

    // ---- ragged calls, clone mid-stream, reset: the same bits ----
    filter::Pfs s(f, M, D);
    std::vector<Complex> part, cat;
    size_t pos = 0;
    for (size_t blk : {1ul, 7ul, 0ul, 100ul}) {
        s.process(y.data() + pos * M, blk, part);
        cat.insert(cat.end(), part.begin(), part.end());
        pos += blk;
    }
    filter::Pfs c(s);
    std::vector<Complex> rest_s, rest_c;
    s.process(y.data() + pos * M, nf - pos, rest_s);
    c.process(y.data() + pos * M, nf - pos, rest_c);
    EXPECT(same_bits(rest_s, rest_c), "clone diverged");
    cat.insert(cat.end(), rest_s.begin(), rest_s.end());
    EXPECT(same_bits(cat, x), "blocked stream differs from one call");
    s.reset();
    std::vector<Complex> again;
    s.process(y.data(), nf, again);
    EXPECT(same_bits(again, x), "reset differs from a fresh handle");

    // ---- channel-major input is the transpose, with the same bits ----
    std::vector<Complex> yt(nf * M);
    for (size_t m = 0; m < nf; ++m)
        for (size_t k = 0; k < M; ++k) yt[k * nf + m] = y[m * M + k];
    filter::Pfs cm(f, M, D, SDR_PFS_CHANNEL_MAJOR);
    std::vector<Complex> xt;
    cm.process(yt.data(), nf, xt);
    EXPECT(same_bits(xt, x), "channel-major input differs");

    // ---- Pfb -> Pfs: the input comes back delayed by L - 1 (Hamming pair: about 50 dB) ----
    const std::vector<float> h = lowpass(12 * (int)M + 1, 0.5 / M, 1.0), fs = lowpass(12 * (int)M + 1, 1.0 / M, (double)D);
    const size_t ns = 200 * M;
    std::vector<Complex> in(ns);
    for (size_t i = 0; i < ns; ++i) in[i] = y[i % y.size()];
    filter::Pfb ana(h, M, D);
    std::vector<Complex> fr, back;
    const size_t fn = ana.process(in.data(), ns, fr);
    filter::Pfs syn(fs, M, D);
    syn.process(fr.data(), fn, back);
    const size_t d = h.size() - 1;
    double pe = 0, pw = 0;
    for (size_t t = 2 * d; t < back.size(); ++t) {
        pw += std::norm(in[t - d]);
        pe += std::norm(back[t] - in[t - d]);
    }
    const double snr = 10 * std::log10(pw / pe);
    EXPECT(back.size() == ns && snr > 40, "round trip: %zu samples, %.1f dB", back.size(), snr);

    if (fails) return 1;
    printf("PFS MIRROR OK (M=%zu D=%zu L=%zu, %zu outputs, max err %.3g of %.3g, round trip %.1f dB)\n", M, D,
           f.size(), n, err, peak, snr);
    return 0;
}

// arb_mirror_test.cpp -- the arbitrary-ratio resampler bank through the C++ host mirror (host/sdr.hpp): filter::Arb
// against the definition evaluated here in f64 at exact 64.64 positions (H(t) interpolated between adjacent phases);
// ragged calls with a different split per channel, clone, set_steps and reset give the bits of one call.  Built and
// run by tests/test_gpu_arb.py (needs a GPU: there is no CPU fallback).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../unnamed-rust-sdr_b200/host/sdr.hpp"

using namespace sdr;
typedef unsigned __int128 u128;

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

static u128 val(sdr_arb_time_t t) { return ((u128)t.whole << 64) | t.frac; }

// z[r] = sum_m H(tau(r) - m) y[m], H(t) = (1 - a) h[j] + a h[j+1], j = floor(t P), a = t P - j, in f64
static std::complex<double> definition(const std::vector<float> &h, size_t P, const Complex *y, u128 tau) {
    const size_t L = h.size();
    const long long n0 = (long long)(tau >> 64);
    std::complex<double> acc(0, 0);
    for (long long m = std::max<long long>(0, n0 - (long long)(L / P) - 2); m <= n0; ++m) {
        const u128 tp = (tau - ((u128)(unsigned long long)m << 64)) * P;
        const unsigned long long j = (unsigned long long)(tp >> 64);
        if (j >= L) continue;
        const double a = (double)(unsigned long long)tp * 0x1p-64;
        const double hj = h[j], hj1 = j + 1 < L ? h[j + 1] : 0.0;
        acc += ((1 - a) * hj + a * hj1) * std::complex<double>(y[m].real(), y[m].imag());
    }
    return acc;
}

int main() {
    const size_t C = 3, P = 64, L = 1024, nf = 3000;
    const std::vector<sdr_arb_time_t> steps = {filter::Arb::step(1.000037, 1.0), filter::Arb::step(48000, 44100),
                                               filter::Arb::step(1.0, 4.41)};
    const std::vector<sdr_arb_time_t> first = {{0, 0}, {2, 0x9E3779B97F4A7C15ull}, {0, 1ull << 63}};
    const std::vector<float> h = lowpass((int)L, 0.4 / P, (double)P);
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i ^ 0xA4B200ull);
        y[i] = Complex((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f, (float)((r >> 8) & 0xFFFF) / 32768.0f - 1.0f);
    }

    // ---- against the definition at exact positions ----
    filter::Arb bank(h, L, P, steps, first);
    std::vector<std::vector<Complex>> z;
    bank.process(y.data(), std::vector<size_t>(C, nf), nf, z);
    double worst = 0;
    for (size_t k = 0; k < C; ++k) {
        const u128 t0 = val(first[k]), st = val(steps[k]), end = (u128)nf << 64;
        const size_t want = t0 >= end ? 0 : (size_t)((end - t0 + st - 1) / st);
        EXPECT(z[k].size() == want, "channel %zu: %zu outputs, want %zu", k, z[k].size(), want);
        double peak = 0, err = 0;
        for (size_t r = 0; r < z[k].size(); ++r) {
            const std::complex<double> ref = definition(h, P, y.data() + k * nf, t0 + (u128)r * st);
            peak = std::max(peak, std::abs(ref));
            err = std::max(err, std::abs(ref - std::complex<double>(z[k][r].real(), z[k][r].imag())));
        }
        EXPECT(err <= 1e-5 * peak, "channel %zu: max |arb - definition| = %g of peak %g", k, err, peak);
        worst = std::max(worst, err / peak);
    }

    // ---- ragged calls, a different split per channel, clone mid-stream, reset: the same bits ----
    filter::Arb s(h, L, P, steps, first);
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
    filter::Arb c(s);
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

    // ---- set_steps after 1000 frames: the outputs before the change are the one-call bits; reset undoes it ----
    s.reset();
    std::vector<std::vector<Complex>> a, b;
    s.process(y.data(), std::vector<size_t>(C, 1000), nf, a);
    s.set_steps({steps[2], steps[0], steps[1]});
    std::vector<Complex> tail(C * nf, Complex(0, 0));
    for (size_t k = 0; k < C; ++k) std::copy(y.begin() + k * nf + 1000, y.begin() + (k + 1) * nf, tail.begin() + k * nf);
    s.process(tail.data(), std::vector<size_t>(C, nf - 1000), nf, b);
    for (size_t k = 0; k < C; ++k) {
        std::vector<Complex> head(z[k].begin(), z[k].begin() + a[k].size());
        EXPECT(same_bits(a[k], head), "channel %zu: outputs before set_steps differ", k);
        EXPECT(!b[k].empty(), "channel %zu: no outputs after set_steps", k);
    }
    s.reset();
    std::vector<std::vector<Complex>> again;
    s.process(y.data(), std::vector<size_t>(C, nf), nf, again);
    for (size_t k = 0; k < C; ++k) EXPECT(same_bits(again[k], z[k]), "channel %zu: reset differs", k);

    if (fails) return 1;
    printf("ARB MIRROR OK (C=%zu P=%zu L=%zu, steps 1.000037 48000/44100 1/4.41, max err %.3g of peak)\n", C, P, L,
           worst);
    return 0;
}

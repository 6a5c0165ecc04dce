// eq_mirror_test.cpp -- the adaptive equalizer bank through the C++ host mirror (host/sdr.hpp): filter::Eq with mu = 0
// and the centre spike delays each row by (N - 1) / 2 symbols bit for bit and keeps its taps; with adaptation, ragged
// calls with a different split per channel, clone and reset give the bits (symbols, errors and taps) of one call.
// Built and run by tests/test_gpu_eq.py (needs a GPU: there is no CPU fallback).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
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

static bool same(const filter::Eq::Out &a, const filter::Eq::Out &b, size_t k, size_t from = 0) {
    const size_t n = a.sym[k].size();
    if (b.sym[k].size() != from + n) return false;
    return std::memcmp(a.sym[k].data(), b.sym[k].data() + from, n * sizeof(Complex)) == 0 &&
           std::memcmp(a.err[k].data(), b.err[k].data() + from, n * sizeof(Complex)) == 0;
}

int main() {
    const size_t C = 3, nf = 3000, N = 11;
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i + 7);
        y[i] = Complex((float)((r & 0xFFFF) / 32768.0 - 1.0), (float)(((r >> 16) & 0xFFFF) / 32768.0 - 1.0));
    }
    const std::vector<size_t> n_all(C, nf);

    // mu = 0, centre spike: y_s = x_{s-5}
    {
        filter::Eq eq(N, C, {{4, 0.f, 1.f, 2.f, ~0ull}});
        const filter::Eq::Out o = eq.process(y.data(), n_all, nf);
        const size_t c = (N - 1) / 2;
        for (size_t k = 0; k < C; ++k) {
            EXPECT(std::memcmp(o.sym[k].data() + c, y.data() + k * nf, (nf - c) * sizeof(Complex)) == 0,
                   "delay ch %zu", k);
            const std::vector<Complex> w = eq.taps(k);
            for (size_t j = 0; j < N; ++j) EXPECT(w[j] == Complex(j == c ? 1.f : 0.f, 0.f), "tap %zu ch %zu", j, k);
        }
    }

    // adapting, one order per channel, CMA then DD at different points
    const std::vector<sdr_eq_adapt_t> adapt = {{2, 0.01f, 1.f, 2.f, 100}, {4, 0.005f, 1.f, 2.f, ~0ull},
                                               {8, 0.02f, 0.8f, 1.f, 0}};
    filter::Eq eq(N, C, adapt);
    const filter::Eq::Out one = eq.process(y.data(), n_all, nf);
    std::vector<std::vector<Complex>> taps(C);
    for (size_t k = 0; k < C; ++k) {
        taps[k] = eq.taps(k);
        bool moved = false;
        for (size_t j = 0; j < N; ++j) moved = moved || taps[k][j] != Complex(j == (N - 1) / 2 ? 1.f : 0.f, 0.f);
        EXPECT(moved, "the taps adapted ch %zu", k);
    }

    // ragged calls, a different split per channel, with a clone halfway; reset
    filter::Eq p(N, C, adapt);
    std::vector<size_t> at(C, 0);
    filter::Eq::Out acc;
    acc.sym.resize(C);
    acc.err.resize(C);
    std::vector<Complex> buf;
    std::unique_ptr<filter::Eq> clone;
    std::vector<size_t> clone_at;
    for (int call = 0; call < 1000; ++call) {
        std::vector<size_t> take(C);
        size_t longest = 0;
        for (size_t k = 0; k < C; ++k) {
            take[k] = std::min<size_t>(nf - at[k], splitmix(call * 7 + k) % 37);
            longest = std::max(longest, take[k]);
        }
        const size_t stride = std::max<size_t>(longest, 1);
        buf.assign(C * stride, Complex(0, 0));
        for (size_t k = 0; k < C; ++k)
            for (size_t j = 0; j < take[k]; ++j) buf[k * stride + j] = y[k * nf + at[k] + j];
        const filter::Eq::Out o = p.process(buf.data(), take, stride);
        for (size_t k = 0; k < C; ++k) {
            acc.sym[k].insert(acc.sym[k].end(), o.sym[k].begin(), o.sym[k].end());
            acc.err[k].insert(acc.err[k].end(), o.err[k].begin(), o.err[k].end());
            at[k] += take[k];
        }
        if (!clone && call == 40) {
            clone.reset(new filter::Eq(p));
            clone_at = at;
        }
    }
    for (size_t k = 0; k < C; ++k) {
        EXPECT(at[k] == nf, "split consumed everything ch %zu", k);
        EXPECT(same(acc, one, k), "ragged calls ch %zu", k);
        EXPECT(p.taps(k) == taps[k], "ragged taps ch %zu", k);
    }
    {
        size_t longest = 0;
        std::vector<size_t> rest(C);
        for (size_t k = 0; k < C; ++k) longest = std::max(longest, rest[k] = nf - clone_at[k]);
        buf.assign(C * longest, Complex(0, 0));
        for (size_t k = 0; k < C; ++k)
            for (size_t j = 0; j < rest[k]; ++j) buf[k * longest + j] = y[k * nf + clone_at[k] + j];
        const filter::Eq::Out o = clone->process(buf.data(), rest, longest);
        for (size_t k = 0; k < C; ++k) {
            EXPECT(same(o, one, k, clone_at[k]), "clone ch %zu", k);
            EXPECT(clone->taps(k) == taps[k], "clone taps ch %zu", k);
        }
    }
    p.reset();
    const filter::Eq::Out again = p.process(y.data(), n_all, nf);
    for (size_t k = 0; k < C; ++k) EXPECT(same(again, one, k), "reset ch %zu", k);

    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("EQ MIRROR OK\n");
    return 0;
}

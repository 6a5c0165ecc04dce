// csync_mirror_test.cpp -- the carrier recovery bank through the C++ host mirror (host/sdr.hpp): filter::Csync with
// kp = ki = 0 advances the phase by exactly 2^24 nu_0 per symbol; with the loop closed, the reported phases follow the
// integer recurrence from the reported errors exactly, and ragged calls with a different split per channel, clone and
// reset give the bits of one call.  Built and run by tests/test_gpu_csync.py (needs a GPU: there is no CPU fallback).
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

static bool same(const filter::Csync::Out &a, const filter::Csync::Out &b, size_t k, size_t from = 0) {
    const size_t n = a.sym[k].size();
    if (b.sym[k].size() != from + n) return false;
    return std::memcmp(a.sym[k].data(), b.sym[k].data() + from, n * sizeof(Complex)) == 0 &&
           std::memcmp(a.phase[k].data(), b.phase[k].data() + from, n * sizeof(uint64_t)) == 0 &&
           std::memcmp(a.err[k].data(), b.err[k].data() + from, n * sizeof(float)) == 0;
}

static long long q40(float x) { return std::llrint((double)x * 0x1p40); }

int main() {
    const size_t C = 3, nf = 3000;
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i + 99);
        y[i] = Complex((float)((r & 0xFFFF) / 32768.0 - 1.0) * 2, (float)(((r >> 16) & 0xFFFF) / 32768.0 - 1.0) * 2);
    }
    const std::vector<size_t> n_all(C, nf);
    const std::vector<uint64_t> phase = {0, 1ull << 63, 0x9E3779B97F4A7C15ull};
    const std::vector<int64_t> freq = {0, 1000000, -123456789};

    // open loop: phi_s = phi_0 + s 2^24 nu_0
    {
        filter::Csync cs(C, {{4, 0.f, 0.f, 1.f, 0.01}}, phase, freq);
        const filter::Csync::Out o = cs.process(y.data(), n_all, nf);
        for (size_t k = 0; k < C; ++k)
            for (size_t s = 0; s < nf; ++s)
                EXPECT(o.phase[k][s] == phase[k] + (uint64_t)s * ((uint64_t)freq[k] << 24), "open loop ch %zu %zu", k,
                       s);
        EXPECT(std::memcmp(o.sym[0].data(), y.data(), nf * sizeof(Complex)) == 0, "phase 0 keeps the symbols");
    }

    // closed loop, one order per channel: the integer recurrence from the reported errors
    const std::vector<sdr_csync_loop_t> loops = {{2, 0.02f, 5e-4f, 1.f, 0.05}, {4, 0.004f, 3e-5f, 2.f, 0.01},
                                                 {8, 0.01f, 1e-4f, 1.5f, 1.0 / 16}};
    filter::Csync cs(C, loops, phase, freq);
    const filter::Csync::Out one = cs.process(y.data(), n_all, nf);
    for (size_t k = 0; k < C; ++k) {
        uint64_t phi = phase[k];
        long long nu = freq[k];
        const long long V = (long long)std::floor(loops[k].max_freq * 0x1p40);
        bool moved = false;
        for (size_t s = 0; s < nf; ++s) {
            EXPECT(one.phase[k][s] == phi, "replay ch %zu symbol %zu", k, s);
            const float e = one.err[k][s];
            moved = moved || e != 0.f;
            const float ie = loops[k].ki * e, pe = loops[k].kp * e;
            nu = std::min(std::max(nu + q40(ie), -V), V);
            phi += (uint64_t)(nu + q40(pe)) << 24;
        }
        EXPECT(moved, "the loop moved ch %zu", k);
        const auto st = cs.state(k);
        EXPECT(st.first == phi && st.second == nu, "state ch %zu", k);
    }

    // ragged calls, a different split per channel, with a clone halfway; reset
    filter::Csync p(C, loops, phase, freq);
    std::vector<size_t> at(C, 0);
    filter::Csync::Out acc;
    acc.sym.resize(C);
    acc.phase.resize(C);
    acc.err.resize(C);
    std::vector<Complex> buf;
    std::unique_ptr<filter::Csync> clone;
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
        const filter::Csync::Out o = p.process(buf.data(), take, stride);
        for (size_t k = 0; k < C; ++k) {
            acc.sym[k].insert(acc.sym[k].end(), o.sym[k].begin(), o.sym[k].end());
            acc.phase[k].insert(acc.phase[k].end(), o.phase[k].begin(), o.phase[k].end());
            acc.err[k].insert(acc.err[k].end(), o.err[k].begin(), o.err[k].end());
            at[k] += take[k];
        }
        if (!clone && call == 40) {
            clone.reset(new filter::Csync(p));
            clone_at = at;
        }
    }
    for (size_t k = 0; k < C; ++k) {
        EXPECT(at[k] == nf, "split consumed everything ch %zu", k);
        EXPECT(same(acc, one, k), "ragged calls ch %zu", k);
    }
    {
        size_t longest = 0;
        std::vector<size_t> rest(C);
        for (size_t k = 0; k < C; ++k) longest = std::max(longest, rest[k] = nf - clone_at[k]);
        buf.assign(C * longest, Complex(0, 0));
        for (size_t k = 0; k < C; ++k)
            for (size_t j = 0; j < rest[k]; ++j) buf[k * longest + j] = y[k * nf + clone_at[k] + j];
        const filter::Csync::Out o = clone->process(buf.data(), rest, longest);
        for (size_t k = 0; k < C; ++k) EXPECT(same(o, one, k, clone_at[k]), "clone ch %zu", k);
    }
    p.reset();
    const filter::Csync::Out again = p.process(y.data(), n_all, nf);
    for (size_t k = 0; k < C; ++k) EXPECT(same(again, one, k), "reset ch %zu", k);

    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("CSYNC MIRROR OK\n");
    return 0;
}

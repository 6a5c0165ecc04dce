// tsync_mirror_test.cpp -- the symbol timing recovery bank through the C++ host mirror (host/sdr.hpp): filter::Tsync
// with kp = ki = 0 gives filter::Arb's outputs and positions bit for bit; with the loop closed, the reported positions
// follow the integer recurrence from the reported errors exactly, and ragged calls with a different split per channel,
// clone and reset give the bits of one call.  Built and run by tests/test_gpu_tsync.py (needs a GPU: there is no CPU
// fallback).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../unnamed-rust-sdr_b200/host/sdr.hpp"

using namespace sdr;
typedef unsigned __int128 u128;
typedef __int128 i128;

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

static u128 val(sdr_arb_time_t t) { return ((u128)t.whole << 64) | t.frac; }

static bool same(const filter::Tsync::Out &a, const filter::Tsync::Out &b, size_t k) {
    if (a.sym[k].size() != b.sym[k].size() || a.pos[k].size() != b.pos[k].size()) return false;
    return std::memcmp(a.sym[k].data(), b.sym[k].data(), a.sym[k].size() * sizeof(Complex)) == 0 &&
           std::memcmp(a.pos[k].data(), b.pos[k].data(), a.pos[k].size() * sizeof(sdr_arb_time_t)) == 0 &&
           std::memcmp(a.err[k].data(), b.err[k].data(), a.err[k].size() * sizeof(float)) == 0;
}

static long long q40(float x) { return std::llrint((double)x * 0x1p40); }

int main() {
    const size_t C = 3, P = 32, L = 511, nf = 3000;
    const std::vector<sdr_arb_time_t> periods = {filter::Arb::step(2.0 * 1.000037, 1.0), filter::Arb::step(4.41, 1.0),
                                                 filter::Arb::step(8.0, 1.0)};
    const std::vector<sdr_arb_time_t> first = {{0, 0}, {2, 0x9E3779B97F4A7C15ull}, {0, 1ull << 63}};
    const std::vector<float> h = lowpass((int)L, 0.4 / P, (double)P);
    std::vector<Complex> y(C * nf);
    for (size_t i = 0; i < C * nf; ++i) {
        const uint64_t r = splitmix(i + 99);
        y[i] = Complex((float)((r & 0xFFFF) / 32768.0 - 1.0) * 2, (float)(((r >> 16) & 0xFFFF) / 32768.0 - 1.0) * 2);
    }
    std::vector<size_t> n_all(C, nf);

    // open loop: Arb at step T and first tau(0)
    {
        filter::Tsync ts(h, L, P, periods, {{0.f, 0.f, 1.f, 0.0}}, first);
        filter::Arb arb(h, L, P, periods, first);
        const filter::Tsync::Out o = ts.process(y.data(), n_all, nf);
        std::vector<std::vector<Complex>> z;
        arb.process(y.data(), n_all, nf, z);
        for (size_t k = 0; k < C; ++k) {
            EXPECT(o.sym[k].size() == z[k].size() && !z[k].empty(), "open-loop count ch %zu", k);
            EXPECT(std::memcmp(o.sym[k].data(), z[k].data(), z[k].size() * sizeof(Complex)) == 0, "open-loop bits %zu",
                   k);
            for (size_t r = 0; r < o.pos[k].size(); ++r)
                EXPECT(val(o.pos[k][r]) == val(first[k]) + (u128)r * val(periods[k]), "open-loop position %zu %zu", k, r);
        }
    }

    // closed loop: the integer recurrence from the reported errors (gains small enough that v never reaches V)
    const std::vector<sdr_tsync_loop_t> loops = {{0.05f, 0.002f, 1.0f, 0.25}};
    filter::Tsync ts(h, L, P, periods, loops, first);
    const filter::Tsync::Out one = ts.process(y.data(), n_all, nf);
    for (size_t k = 0; k < C; ++k) {
        u128 tau = val(first[k]);
        long long v = 0;
        const u128 T = val(periods[k]);
        bool moved = false;
        for (size_t s = 0; s < one.pos[k].size(); ++s) {
            EXPECT(val(one.pos[k][s]) == tau, "replay ch %zu symbol %zu", k, s);
            const float e = one.err[k][s];
            moved = moved || e != 0.f;
            const float ie = loops[0].ki * e, pe = loops[0].kp * e;
            v -= q40(ie);
            EXPECT(std::fabs((double)v) < 0.25 * (double)T * 0x1p-24, "v stays inside V");
            tau = (u128)((i128)tau + (i128)T + ((i128)(v - q40(pe)) << 24));
        }
        EXPECT(moved, "the loop moved ch %zu", k);
        const auto st = ts.state(k);
        EXPECT(val(st.first) == tau && st.second == v, "state ch %zu", k);
    }

    // ragged calls, a different split per channel, with a clone halfway; reset
    filter::Tsync p(h, L, P, periods, loops, first);
    std::vector<size_t> at(C, 0);
    filter::Tsync::Out acc;
    acc.sym.resize(C);
    acc.pos.resize(C);
    acc.err.resize(C);
    std::vector<Complex> buf;
    std::unique_ptr<filter::Tsync> clone;
    std::vector<size_t> clone_at, clone_made;
    for (int call = 0; call < 1000; ++call) {
        std::vector<size_t> take(C);
        size_t longest = 0;
        for (size_t k = 0; k < C; ++k) {
            take[k] = std::min<size_t>(nf - at[k], splitmix(call * 7 + k) % 37);
            longest = std::max(longest, take[k]);
        }
        buf.assign(C * std::max<size_t>(longest, 1), Complex(0, 0));
        for (size_t k = 0; k < C; ++k)
            for (size_t j = 0; j < take[k]; ++j) buf[k * std::max<size_t>(longest, 1) + j] = y[k * nf + at[k] + j];
        const filter::Tsync::Out o = p.process(buf.data(), take, std::max<size_t>(longest, 1));
        for (size_t k = 0; k < C; ++k) {
            acc.sym[k].insert(acc.sym[k].end(), o.sym[k].begin(), o.sym[k].end());
            acc.pos[k].insert(acc.pos[k].end(), o.pos[k].begin(), o.pos[k].end());
            acc.err[k].insert(acc.err[k].end(), o.err[k].begin(), o.err[k].end());
            at[k] += take[k];
        }
        if (!clone && call == 40) {
            clone.reset(new filter::Tsync(p));
            clone_at = at;
            for (size_t k = 0; k < C; ++k) clone_made.push_back(acc.sym[k].size());
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
        const filter::Tsync::Out o = clone->process(buf.data(), rest, longest);
        for (size_t k = 0; k < C; ++k)
            EXPECT(o.sym[k].size() == one.sym[k].size() - clone_made[k] &&
                       std::memcmp(o.sym[k].data(), one.sym[k].data() + clone_made[k],
                                   o.sym[k].size() * sizeof(Complex)) == 0,
                   "clone ch %zu", k);
    }
    p.reset();
    const filter::Tsync::Out again = p.process(y.data(), n_all, nf);
    for (size_t k = 0; k < C; ++k) EXPECT(same(again, one, k), "reset ch %zu", k);

    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("TSYNC MIRROR OK\n");
    return 0;
}

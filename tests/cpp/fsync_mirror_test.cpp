// fsync_mirror_test.cpp -- the frame synchronizer bank through the C++ host mirror (host/sdr.hpp): fec::Fsync on three
// channels of framed QPSK, each turned by its own quarter turns, finds every frame at its word, reports the rotation and
// emits payloads equal to the transmitted symbols exactly; ragged calls with a different split per channel, clone and
// reset give the bits of one call.  Built and run by tests/test_gpu_fsync.py (needs a GPU: there is no CPU fallback).
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

static Complex qpsk(uint64_t r) {
    const float a = 0.70710678f;
    return Complex(r & 1 ? -a : a, r & 2 ? -a : a);
}

// x i^q, exactly
static Complex turn(Complex x, unsigned q) {
    for (unsigned i = 0; i < q % 4; ++i) x = Complex(-x.imag(), x.real());
    return x;
}

static bool same(const fec::Fsync::Out &a, const fec::Fsync::Out &b, size_t k) {
    return a.payload[k].size() == b.payload[k].size() && a.records[k].size() == b.records[k].size() &&
           std::memcmp(a.payload[k].data(), b.payload[k].data(), a.payload[k].size() * sizeof(Complex)) == 0 &&
           std::memcmp(a.records[k].data(), b.records[k].data(), a.records[k].size() * sizeof(sdr_fsync_record_t)) == 0;
}

int main() {
    const size_t C = 3, Lp = 32, F = 32 + 300, frames = 12, lead = 77, n = lead + frames * F;
    std::vector<Complex> word(Lp);
    for (size_t j = 0; j < Lp; ++j) word[j] = qpsk(splitmix(j + 1));
    std::vector<Complex> y(C * n), sent(C * n);
    for (size_t k = 0; k < C; ++k)
        for (size_t i = 0; i < n; ++i) {
            const size_t f = (i - lead) % F;
            sent[k * n + i] = i >= lead && f < Lp ? word[f] : qpsk(splitmix(1000 + k * n + i));
            y[k * n + i] = turn(sent[k * n + i], (unsigned)k + 1);
        }
    const std::vector<size_t> n_all(C, n);
    const std::vector<sdr_fsync_params_t> params = {{(uint32_t)F, 4, 0.5f, 0.3f, 1, 2, 2}};
    fec::Fsync fs(C, Lp, word, params);
    const fec::Fsync::Out one = fs.process(y.data(), n_all, n);
    for (size_t k = 0; k < C; ++k) {
        size_t emitted = 0;
        for (const sdr_fsync_record_t &r : one.records[k]) {
            EXPECT((r.pos - lead) % F == 0, "ch %zu record at %llu", k, (unsigned long long)r.pos);
            if (r.out_index == UINT64_MAX) continue;
            ++emitted;
            EXPECT(r.rot == (k + 1) % 4, "ch %zu rot %u", k, (unsigned)r.rot);
            for (size_t j = 0; j < F - Lp && r.out_index + j < one.payload[k].size(); ++j)
                EXPECT(one.payload[k][r.out_index + j] == sent[k * n + r.pos + Lp + j], "ch %zu payload %zu", k, j);
        }
        EXPECT(emitted == frames - 1, "ch %zu: %zu frames emitted", k, emitted);  // frame 0 is the HIT
        const sdr_fsync_state_t st = fs.state(k);
        EXPECT(st.state == SDR_FSYNC_LOCK && st.consumed == n, "ch %zu state", k);
    }

    // ragged calls, a different split per channel, with a clone halfway; reset
    fec::Fsync p(C, Lp, word, params);
    std::vector<size_t> at(C, 0);
    fec::Fsync::Out acc;
    acc.payload.resize(C);
    acc.records.resize(C);
    std::vector<Complex> buf;
    std::unique_ptr<fec::Fsync> clone;
    fec::Fsync::Out cacc;
    cacc.payload.resize(C);
    cacc.records.resize(C);
    auto add = [&](fec::Fsync::Out &to, const fec::Fsync::Out &o) {
        for (size_t k = 0; k < C; ++k) {
            to.payload[k].insert(to.payload[k].end(), o.payload[k].begin(), o.payload[k].end());
            to.records[k].insert(to.records[k].end(), o.records[k].begin(), o.records[k].end());
        }
    };
    for (int call = 0; call < 100000 && (at[0] < n || at[1] < n || at[2] < n); ++call) {
        std::vector<size_t> take(C);
        size_t longest = 0;
        for (size_t k = 0; k < C; ++k) {
            take[k] = std::min<size_t>(n - at[k], splitmix(call * 7 + k) % 97);
            longest = std::max(longest, take[k]);
        }
        const size_t stride = std::max<size_t>(longest, 1);
        buf.assign(C * stride, Complex(0, 0));
        for (size_t k = 0; k < C; ++k)
            for (size_t j = 0; j < take[k]; ++j) buf[k * stride + j] = y[k * n + at[k] + j];
        const fec::Fsync::Out o = p.process(buf.data(), take, stride);
        add(acc, o);
        if (clone) add(cacc, clone->process(buf.data(), take, stride));
        if (!clone && call == 20) {
            clone.reset(new fec::Fsync(p));
            cacc = acc;
        }
        for (size_t k = 0; k < C; ++k) at[k] += take[k];
    }
    for (size_t k = 0; k < C; ++k) {
        EXPECT(same(acc, one, k), "ragged calls ch %zu", k);
        EXPECT(same(cacc, one, k), "clone ch %zu", k);
    }
    p.reset();
    const fec::Fsync::Out again = p.process(y.data(), n_all, n);
    for (size_t k = 0; k < C; ++k) EXPECT(same(again, one, k), "reset ch %zu", k);

    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("FSYNC MIRROR OK\n");
    return 0;
}

// vit_mirror_test.cpp -- the Viterbi decoder bank through the C++ host mirror (host/sdr.hpp): fec::Vit decodes noiseless
// K = 7 rate-1/2 codewords (zero-tailed messages) to their messages through process and a terminated finish; ragged
// calls with a different split per channel, a clone halfway and reset give the bits of one call.
// Built and run by tests/test_gpu_vit.py (needs a GPU: there is no CPU fallback).
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

int main() {
    const unsigned K = 7;
    const std::vector<uint32_t> gens = {0133, 0171};
    const size_t C = 3, m = 2000, L = 64, n = 2;
    // messages with K - 1 zero tail bits, their codewords as soft values +-0.5 and, on channel 1, noise of +-0.3
    std::vector<uint8_t> msg(C * m);
    std::vector<float> x(C * m * n);
    for (size_t k = 0; k < C; ++k) {
        uint32_t s = 0;
        for (size_t t = 0; t < m; ++t) {
            const uint32_t u = t + K - 1 < m ? (uint32_t)(splitmix(k * m + t) & 1) : 0;
            msg[k * m + t] = (uint8_t)u;
            const uint32_t r = (u << (K - 1)) | s;
            for (size_t j = 0; j < n; ++j) {
                const float c = (float)(__builtin_popcount(r & gens[j]) & 1);
                float v = 0.5f * (1.f - 2.f * c);
                if (k == 1) v += 0.3f * (float)((double)(splitmix(1000003 + t * n + j) % 2001) / 1000.0 - 1.0);
                x[(k * m + t) * n + j] = v;
            }
            s = r >> 1;
        }
    }
    const std::vector<size_t> n_all(C, m);
    fec::Vit v(K, gens, L, {100.f}, C);
    std::vector<std::vector<uint8_t>> one = v.process(x.data(), n_all, m);
    const std::vector<std::vector<uint8_t>> tail = v.finish(true);
    for (size_t k = 0; k < C; ++k) {
        EXPECT(one[k].size() == (m & ~(size_t)31) - L, "count ch %zu: %zu", k, one[k].size());
        one[k].insert(one[k].end(), tail[k].begin(), tail[k].end());
        EXPECT(one[k].size() == m && std::memcmp(one[k].data(), msg.data() + k * m, m) == 0, "decode ch %zu", k);
    }

    // ragged calls, a different split per channel, with a clone halfway; reset
    fec::Vit p(K, gens, L, {100.f}, C);
    std::vector<size_t> at(C, 0);
    std::vector<std::vector<uint8_t>> acc(C);
    std::vector<float> buf;
    std::unique_ptr<fec::Vit> clone;
    std::vector<size_t> clone_at, clone_got;
    for (int call = 0; call < 400; ++call) {
        std::vector<size_t> take(C);
        size_t longest = 0;
        for (size_t k = 0; k < C; ++k) {
            take[k] = std::min<size_t>(m - at[k], splitmix(call * 7 + k) % 45);
            longest = std::max(longest, take[k]);
        }
        const size_t stride = std::max<size_t>(longest, 1);
        buf.assign(C * stride * n, 0.f);
        for (size_t k = 0; k < C; ++k)
            std::memcpy(&buf[k * stride * n], &x[(k * m + at[k]) * n], take[k] * n * sizeof(float));
        const std::vector<std::vector<uint8_t>> o = p.process(buf.data(), take, stride);
        for (size_t k = 0; k < C; ++k) {
            acc[k].insert(acc[k].end(), o[k].begin(), o[k].end());
            at[k] += take[k];
        }
        if (!clone && call == 20) {
            clone.reset(new fec::Vit(p));
            clone_at = at;
            for (size_t k = 0; k < C; ++k) clone_got.push_back(acc[k].size());
        }
    }
    const std::vector<std::vector<uint8_t>> ptail = p.finish(true);
    for (size_t k = 0; k < C; ++k) {
        EXPECT(at[k] == m, "split consumed everything ch %zu", k);
        acc[k].insert(acc[k].end(), ptail[k].begin(), ptail[k].end());
        EXPECT(acc[k] == one[k], "ragged calls ch %zu", k);
    }
    {
        size_t longest = 0;
        std::vector<size_t> rest(C);
        for (size_t k = 0; k < C; ++k) longest = std::max(longest, rest[k] = m - clone_at[k]);
        buf.assign(C * longest * n, 0.f);
        for (size_t k = 0; k < C; ++k)
            std::memcpy(&buf[k * longest * n], &x[(k * m + clone_at[k]) * n], rest[k] * n * sizeof(float));
        std::vector<std::vector<uint8_t>> o = clone->process(buf.data(), rest, longest);
        const std::vector<std::vector<uint8_t>> ct = clone->finish(true);
        for (size_t k = 0; k < C; ++k) {
            o[k].insert(o[k].end(), ct[k].begin(), ct[k].end());
            EXPECT(clone_got[k] + o[k].size() == m &&
                       std::memcmp(o[k].data(), one[k].data() + clone_got[k], o[k].size()) == 0,
                   "clone ch %zu", k);
        }
    }
    p.reset();
    std::vector<std::vector<uint8_t>> again = p.process(x.data(), n_all, m);
    const std::vector<std::vector<uint8_t>> at2 = p.finish(true);
    for (size_t k = 0; k < C; ++k) {
        again[k].insert(again[k].end(), at2[k].begin(), at2[k].end());
        EXPECT(again[k] == one[k], "reset ch %zu", k);
    }

    if (fails) {
        printf("%d failures\n", fails);
        return 1;
    }
    printf("VIT MIRROR OK\n");
    return 0;
}

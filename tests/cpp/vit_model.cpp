// vit_model.cpp -- the sdr_vit definition (tests/vit_ref.py) restated in C++ for one channel, for streams too long for
// the numpy model: exact int64 metrics, never renormalised.  tests/test_vit_host.py checks it against vit_ref.model on
// short streams; tests/test_gpu_vit.py uses it where the least metric passes 2^32.
//     vit_model K L zero_start scale g_0 .. g_{n-1} in.f32 out.u8
// reads the n f32 soft values of every step, writes the released bits and prints the least final metric.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

int main(int argc, char **argv) {
    if (argc < 9) {
        fprintf(stderr, "usage: vit_model K L zero_start scale g_0 .. g_{n-1} in.f32 out.u8\n");
        return 2;
    }
    const int K = atoi(argv[1]), L = atoi(argv[2]), zs = atoi(argv[3]);
    const float sigma = (float)atof(argv[4]);
    const int n = argc - 7;
    std::vector<uint32_t> g(n);
    for (int j = 0; j < n; ++j) g[j] = (uint32_t)strtoul(argv[5 + j], nullptr, 0);
    FILE *f = fopen(argv[5 + n], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END);
    const long bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<float> x(bytes / 4);
    if (fread(x.data(), 4, x.size(), f) != x.size()) return 2;
    fclose(f);
    const int S = 1 << (K - 1), R = L + 32;
    const long long T = (long long)x.size() / n;
    std::vector<int> pat[2];
    for (int b = 0; b < 2; ++b) {
        pat[b].resize(S);
        for (int s = 0; s < S; ++s) {
            const uint32_t r = ((uint32_t)(s >> (K - 2)) << (K - 1)) | ((uint32_t)(s << 1) & (S - 1)) | b;
            int p = 0;
            for (int j = 0; j < n; ++j) p |= (__builtin_popcount(r & g[j]) & 1) << j;
            pat[b][s] = p;
        }
    }
    const long long I = (long long)(K - 1) * 254 * n + 1;
    std::vector<long long> m(S, zs ? I : 0), mn(S);
    m[0] = 0;
    std::vector<uint8_t> dec((size_t)R * S), out;
    std::vector<long long> cost(1 << n);
    for (long long t = 0; t < T; ++t) {
        int q[4] = {0, 0, 0, 0};
        for (int j = 0; j < n; ++j) {
            const float v = x[t * n + j];
            if (std::isfinite(v)) q[j] = (int)std::nearbyint(std::min(std::max(v * sigma, -127.f), 127.f));
        }
        for (int p = 0; p < (1 << n); ++p) {
            long long c = 0;
            for (int j = 0; j < n; ++j) c += ((p >> j) & 1) ? 127 + q[j] : 127 - q[j];
            cost[p] = c;
        }
        uint8_t *d = &dec[(size_t)(t % R) * S];
        for (int s = 0; s < S; ++s) {
            const int p0 = (s << 1) & (S - 1);
            const long long a0 = m[p0] + cost[pat[0][s]], a1 = m[p0 | 1] + cost[pat[1][s]];
            d[s] = a1 < a0;
            mn[s] = a1 < a0 ? a1 : a0;
        }
        m.swap(mn);
        const long long Tn = t + 1;
        if (Tn % 32 == 0 && Tn >= L + 32) {
            int s = (int)(std::min_element(m.begin(), m.end()) - m.begin());
            uint8_t bits[32];
            for (long long i = Tn - 1; i >= Tn - L - 32; --i) {
                if (i < Tn - L) bits[i - (Tn - L - 32)] = (uint8_t)(s >> (K - 2));
                s = ((s << 1) & (S - 1)) | dec[(size_t)(i % R) * S + s];
            }
            out.insert(out.end(), bits, bits + 32);
        }
    }
    f = fopen(argv[6 + n], "wb");
    if (!f || fwrite(out.data(), 1, out.size(), f) != out.size()) return 2;
    fclose(f);
    printf("%lld\n", *std::min_element(m.begin(), m.end()));
    return 0;
}

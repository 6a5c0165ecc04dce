// fsync.cu -- K19, sdr_fsync_*: frame synchronizer bank.  C independent c64 symbol streams; channel k has a sync word
// p of Lp symbols (one Lp per handle) and {F, M, th_search, th_check, V, max_miss, W}.  Position s correlates the word
// with z_s .. z_{s+Lp-1}:
//     c_s = sum_j conj(p_j) z_{s+j},  E_s = sum_j |z_{s+j}|^2,  rho_s = |c_s|^2 / (E_s E_p)   (0 unless E_s E_p > 0)
// with every f32 operation rounded on its own and both sums sequential in j (include/sdr_b200.h states each
// operation), so a numpy float32 restatement gives every c and rho bit for bit.  A search -> verify -> lock ->
// flywheel state machine over the positions decides where frames start; each emitted frame's payload
// z_{s+Lp} .. z_{s+F-1} is derotated by the rotation R read from the phase of its correlation.
// One warp owns one channel and runs its state machine with every lane holding the same state: a search round
// correlates 32 consecutive positions (one per lane) and takes the first hit by ballot; a check correlates the 2W + 1
// window positions and reduces to the best by shuffles; payloads stream through the warp.  The word and the symbols
// of a round sit in shared memory.  Symbols before the call come from a carried tail (fewer than Lp + 2 W symbols),
// read through two pointers as bank.cuh does; the kernel itself writes the next call's tail into the other buffer.
// Counts depend on the data, so a call copies the C counts back before it returns.
#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"

using namespace sdr;

namespace {

constexpr size_t FS_MAX_CH = 65536;
constexpr size_t FS_MIN_LP = 8, FS_MAX_LP = 1024;
constexpr unsigned FS_MAX_F = 1u << 24, FS_MAX_W = 32, FS_MAX_V = 8, FS_MAX_MISS = 255;
constexpr unsigned long long FS_MAX_POS = 1ull << 62;  // symbol totals stay below
constexpr int FS_WARPS = 4;                            // channels (warps) per CTA
constexpr size_t FS_HOST_BYTES = (size_t)32 << 20;    // host-memory calls: chunk size of input
constexpr unsigned long long FS_NONE = ~0ull;

struct FsChan {                 // per channel, fixed at create
    long long word;             // offset (float2 entries) of the channel's word
    long long tail;             // offset of the channel's carried symbols in a tail buffer (Lp + 2W entries)
    float Ep, ths, thc;         // E_p, th_search, th_check
    unsigned F, M, V, mm, W;
};

struct FsState {                // per channel, on the device between calls
    unsigned long long pos;     // sigma (SEARCH) or e
    unsigned long long consumed;
    unsigned long long payload;
    unsigned long long fnext, fend;  // the frame being emitted: next symbol, end (fnext == fend: none)
    unsigned state, cnt, R, ncarry;  // ncarry: the tail holds symbols [consumed - ncarry, consumed)
};

// smem per warp: the word (Lp) and one round's symbols (32 + Lp - 1, padded to 32 + Lp)
inline size_t fs_smem(size_t Lp) { return (size_t)FS_WARPS * (2 * Lp + 32) * sizeof(float2); }

__device__ __forceinline__ unsigned fs_rot(float cr, float ci, unsigned M, float K) {
    if (M == 2) return cr >= 0.f ? 0u : 1u;
    const unsigned q = fabsf(cr) >= fabsf(ci) ? (cr >= 0.f ? 0u : 2u) : (ci >= 0.f ? 1u : 3u);
    if (M == 4) return q;
    float re = cr, im = ci;  // c (-i)^q
    if (q & 2) {
        re = -re;
        im = -im;
    }
    if (q & 1) {
        const float t = re;
        re = im;
        im = -t;
    }
    const float t = __fmul_rn(K, re);
    const int o = im > t ? 1 : (im < -t ? -1 : 0);
    return (unsigned)((int)(2 * q) + o) & 7u;
}

__device__ __forceinline__ float2 fs_derot(float2 x, unsigned r, unsigned M, float h) {
    unsigned q = r;
    if (M == 2) {
        q = 2 * r;
    } else if (M == 8) {
        if (r & 1) x = make_float2(__fmul_rn(__fadd_rn(x.x, x.y), h), __fmul_rn(__fsub_rn(x.y, x.x), h));
        q = r >> 1;
    }
    if (q & 2) x = make_float2(-x.x, -x.y);
    if (q & 1) x = make_float2(x.y, -x.x);
    return x;
}

// a better than b: larger key (rho, NaN as -1; -2 for no position), then nearer e, then earlier
__device__ __forceinline__ bool fs_better(float ka, long long da, long long sa, float kb, long long db, long long sb) {
    return ka > kb || (ka == kb && (da < db || (da == db && sa < sb)));
}

__global__ void __launch_bounds__(FS_WARPS * 32) fsync_kernel(const FsChan *__restrict__ chans,
                                                              const float2 *__restrict__ words, FsState *state,
                                                              const long long *__restrict__ n_in, int C, int Lp,
                                                              float K, float h, const float2 *__restrict__ tail_old,
                                                              float2 *__restrict__ tail_new,
                                                              const float2 *__restrict__ in, long long in_stride,
                                                              float2 *__restrict__ out, long long out_stride,
                                                              sdr_fsync_record_t *__restrict__ recs,
                                                              long long rec_stride, long long *__restrict__ counts) {
    extern __shared__ float2 fs_smem_buf[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = blockIdx.x * FS_WARPS + warp;
    if (k >= C) return;  // whole warps; no CTA barrier follows
    float2 *s_word = fs_smem_buf + (size_t)warp * (2 * Lp + 32);
    float2 *s_z = s_word + Lp;
    const FsChan ch = chans[k];
    for (int j = lane; j < Lp; j += 32) s_word[j] = __ldg(words + ch.word + j);
    FsState st = state[k];
    const unsigned long long T0 = st.consumed, Tend = T0 + (unsigned long long)n_in[k];
    const unsigned long long base = T0 - st.ncarry;
    const float2 *row = in + k * in_stride;
    const float2 *tl = tail_old + ch.tail;
    auto sym = [&](unsigned long long t) -> float2 { return t >= T0 ? __ldg(row + (t - T0)) : tl[t - base]; };
    float2 *orow = out + k * out_stride;
    sdr_fsync_record_t *rrow = recs ? recs + k * rec_stride : nullptr;
    unsigned long long nout = 0, nrec = 0;
    const unsigned long long Lq = (unsigned long long)Lp;

    // c and rho at position s0 + lane for lanes below cnt (every symbol they read has arrived)
    auto correlate = [&](unsigned long long s0, int cnt, float &cr, float &ci, float &rho) {
        __syncwarp();
        for (int i = lane; i < cnt + Lp - 1; i += 32) s_z[i] = sym(s0 + i);
        __syncwarp();
        cr = ci = rho = 0.f;
        if (lane < cnt) {
            const float2 *zz = s_z + lane;
            float2 p = s_word[0], z = zz[0];
            cr = __fadd_rn(__fmul_rn(p.x, z.x), __fmul_rn(p.y, z.y));
            ci = __fsub_rn(__fmul_rn(p.x, z.y), __fmul_rn(p.y, z.x));
            float es = __fadd_rn(__fmul_rn(z.x, z.x), __fmul_rn(z.y, z.y));
#pragma unroll 4
            for (int j = 1; j < Lp; ++j) {
                p = s_word[j];
                z = zz[j];
                cr = __fadd_rn(cr, __fadd_rn(__fmul_rn(p.x, z.x), __fmul_rn(p.y, z.y)));
                ci = __fadd_rn(ci, __fsub_rn(__fmul_rn(p.x, z.y), __fmul_rn(p.y, z.x)));
                es = __fadd_rn(es, __fadd_rn(__fmul_rn(z.x, z.x), __fmul_rn(z.y, z.y)));
            }
            const float a = __fadd_rn(__fmul_rn(cr, cr), __fmul_rn(ci, ci)), b = __fmul_rn(es, ch.Ep);
            rho = b > 0.f ? __fdiv_rn(a, b) : 0.f;
        }
    };
    auto record = [&](unsigned long long pos, unsigned long long oi, float cr, float ci, float rho, unsigned rot,
                      unsigned kind) {
        if (rrow && lane == 0) {
            sdr_fsync_record_t r;
            r.pos = pos;
            r.out_index = oi;
            r.corr[0] = cr;
            r.corr[1] = ci;
            r.rho = rho;
            r.rot = (uint16_t)rot;
            r.kind = (uint16_t)kind;
            rrow[nrec] = r;
        }
        ++nrec;
    };
    auto emit = [&](unsigned long long s) -> unsigned long long {
        st.fnext = s + Lq;
        st.fend = s + ch.F;
        const unsigned long long at = st.payload;
        st.payload += ch.F - Lq;
        return at;
    };

    for (;;) {
        if (st.fnext < st.fend) {  // the frame being emitted: its symbols that have arrived
            const unsigned long long b = min(st.fend, Tend);
            for (unsigned long long t = st.fnext + lane; t < b; t += 32)
                orow[nout + (t - st.fnext)] = fs_derot(sym(t), st.R, ch.M, h);
            if (b > st.fnext) {
                nout += b - st.fnext;
                st.fnext = b;
            }
            if (st.fnext < st.fend) break;  // the next decision needs later symbols anyway
        }
        float cr, ci, rho;
        if (st.state == SDR_FSYNC_SEARCH) {
            if (st.pos + Lq > Tend) break;
            const unsigned long long s0 = st.pos;
            const int cnt = (int)min(32ull, Tend - Lq + 1 - s0);
            correlate(s0, cnt, cr, ci, rho);
            const unsigned hit = __ballot_sync(0xffffffffu, lane < cnt && rho >= ch.ths);
            if (!hit) {
                st.pos = s0 + cnt;
                continue;
            }
            const int l = __ffs(hit) - 1;
            cr = __shfl_sync(0xffffffffu, cr, l);
            ci = __shfl_sync(0xffffffffu, ci, l);
            rho = __shfl_sync(0xffffffffu, rho, l);
            const unsigned long long s = s0 + l;
            const unsigned r = fs_rot(cr, ci, ch.M, K);
            if (ch.V == 0) {
                st.R = r;
                record(s, emit(s), cr, ci, rho, r, SDR_FSYNC_HIT);
                st.state = SDR_FSYNC_LOCK;
            } else {
                record(s, FS_NONE, cr, ci, rho, r, SDR_FSYNC_HIT);
                st.state = SDR_FSYNC_VERIFY;
            }
            st.cnt = 0;
            st.pos = s + ch.F;
            continue;
        }
        const unsigned long long e = st.pos;
        if (e + ch.W + Lq > Tend) break;
        // the best position of the window: per lane over the rounds, then across the warp
        float bk = -2.f, bcr = 0.f, bci = 0.f, brho = 0.f;
        long long bd = 1ll << 40, bs = 0;
        for (unsigned long long s0 = e - ch.W; s0 <= e + ch.W; s0 += 32) {
            const int cnt = (int)min(32ull, e + ch.W + 1 - s0);
            correlate(s0, cnt, cr, ci, rho);
            if (lane < cnt) {
                const long long s = (long long)(s0 + lane), d = s > (long long)e ? s - (long long)e : (long long)e - s;
                const float key = rho != rho ? -1.f : rho;
                if (fs_better(key, d, s, bk, bd, bs)) {
                    bk = key;
                    bd = d;
                    bs = s;
                    bcr = cr;
                    bci = ci;
                    brho = rho;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ok = __shfl_xor_sync(0xffffffffu, bk, o);
            const long long od = __shfl_xor_sync(0xffffffffu, bd, o), os = __shfl_xor_sync(0xffffffffu, bs, o);
            const float ocr = __shfl_xor_sync(0xffffffffu, bcr, o), oci = __shfl_xor_sync(0xffffffffu, bci, o);
            const float orho = __shfl_xor_sync(0xffffffffu, brho, o);
            if (fs_better(ok, od, os, bk, bd, bs)) {
                bk = ok;
                bd = od;
                bs = os;
                bcr = ocr;
                bci = oci;
                brho = orho;
            }
        }
        const unsigned long long s = (unsigned long long)bs;
        const bool pass = brho >= ch.thc;
        const unsigned r = fs_rot(bcr, bci, ch.M, K);
        if (st.state == SDR_FSYNC_VERIFY) {
            if (pass) {
                if (++st.cnt == ch.V) {
                    st.R = r;
                    record(s, emit(s), bcr, bci, brho, r, SDR_FSYNC_VERIFY_PASS);
                    st.state = SDR_FSYNC_LOCK;
                    st.cnt = 0;
                } else {
                    record(s, FS_NONE, bcr, bci, brho, r, SDR_FSYNC_VERIFY_PASS);
                }
                st.pos = s + ch.F;
            } else {
                record(e, FS_NONE, bcr, bci, brho, r, SDR_FSYNC_VERIFY_FAIL);
                st.state = SDR_FSYNC_SEARCH;
                st.pos = e + ch.W + 1;
                st.cnt = 0;
            }
        } else if (pass) {
            st.R = r;
            record(s, emit(s), bcr, bci, brho, r, SDR_FSYNC_LOCK_PASS);
            st.cnt = 0;
            st.pos = s + ch.F;
        } else if (++st.cnt < ch.mm) {
            record(e, emit(e), bcr, bci, brho, st.R, SDR_FSYNC_LOCK_MISS);
            st.pos = e + ch.F;
        } else {
            record(e, FS_NONE, bcr, bci, brho, r, SDR_FSYNC_LOCK_LOST);
            st.state = SDR_FSYNC_SEARCH;
            st.pos = e + ch.W + 1;
            st.cnt = 0;
        }
    }
    // the next call's tail: every symbol from the first one a pending decision reads
    const unsigned long long need = st.state == SDR_FSYNC_SEARCH ? st.pos : st.pos - ch.W;
    const unsigned long long keep = max(base, min(need, Tend));
    for (unsigned long long t = keep + lane; t < Tend; t += 32) tail_new[ch.tail + (t - keep)] = sym(t);
    st.ncarry = (unsigned)(Tend - keep);
    st.consumed = Tend;
    if (lane == 0) {
        state[k] = st;
        counts[k] = (long long)nout;
        counts[C + k] = (long long)nrec;
    }
}

// E_p: the sequential f32 sum of fl(fl(re re) + fl(im im)) (host floats are IEEE single, nothing contracted)
float word_energy(const float *p, size_t Lp) {
    float e = 0.f;
    for (size_t j = 0; j < Lp; ++j) {
        const float re = p[2 * j], im = p[2 * j + 1];
        const float term = re * re + im * im;
        e = j ? e + term : term;
    }
    return e;
}

}  // namespace

struct FsyncHost {
    int dev = 0;
    size_t C = 0, Lp = 0;
    std::vector<FsChan> chans;
    std::vector<float2> words;
    size_t tail_len = 0;                    // sum of Lp + 2W
    std::vector<unsigned long long> total;  // symbols consumed, per channel
    bool fresh = true;                      // the device state is the creation state's once uploaded
};

struct sdr_fsync : FsyncHost {
    StreamRef stream;
    DevBuf d_chans, d_words, d_state, d_n, d_tail[2];
    int cur = 0;
    std::vector<long long> n_host, cnt_host;
    DevBuf d_in, d_out, d_rec;

    int alloc(void *user_stream, const sdr_fsync *) {
        int rc = stream.init(user_stream);
        if (rc) return rc;
        if ((rc = d_chans.upload(chans.data(), C * sizeof(FsChan), stream.s))) return rc;
        if ((rc = d_words.upload(words.data(), words.size() * sizeof(float2), stream.s))) return rc;
        if ((rc = d_state.alloc(C * sizeof(FsState)))) return rc;
        if ((rc = d_n.alloc(C * 3 * sizeof(long long)))) return rc;  // n_in, then the 2C counts
        for (int i = 0; i < 2; ++i)
            if ((rc = d_tail[i].alloc(tail_len * sizeof(float2)))) return rc;
        // one attribute per device shared by every handle: the largest footprint admits every word length
        SDR_CUDA_TRY(cudaFuncSetAttribute(fsync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)fs_smem(FS_MAX_LP)));
        return cuda_status(cudaStreamSynchronize(stream.s));
    }
    int copy_device(const sdr_fsync &src) {
        SDR_CUDA_TRY(cudaMemcpy(d_state.p, src.d_state.p, C * sizeof(FsState), cudaMemcpyDeviceToDevice));
        return cuda_status(
            cudaMemcpy(d_tail[0].p, src.d_tail[src.cur].p, tail_len * sizeof(float2), cudaMemcpyDeviceToDevice));
    }
};

extern "C" sdr_fsync_t *sdr_fsync_create(const sdr_fsync_config_t *cfg, int *err) {
    bool ok = cfg && cfg->words && cfg->params && cfg->word_len >= FS_MIN_LP && cfg->word_len <= FS_MAX_LP &&
              cfg->n_channels >= 1 && cfg->n_channels <= FS_MAX_CH &&
              (cfg->n_words == 1 || cfg->n_words == cfg->n_channels) &&
              (cfg->n_params == 1 || cfg->n_params == cfg->n_channels);
    const size_t Lp = ok ? cfg->word_len : 0;
    std::vector<float> Ep;
    for (size_t w = 0; ok && w < cfg->n_words; ++w) {
        const float *p = cfg->words + 2 * w * Lp;
        for (size_t j = 0; ok && j < 2 * Lp; ++j) ok = std::isfinite(p[j]);
        if (!ok) break;
        Ep.push_back(word_energy(p, Lp));
        ok = Ep.back() > 0.f && std::isfinite(Ep.back());
    }
    for (size_t i = 0; ok && i < cfg->n_params; ++i) {
        const sdr_fsync_params_t &q = cfg->params[i];
        ok = (q.order == 2 || q.order == 4 || q.order == 8) && q.thresh_search > 0.f && q.thresh_search <= 1.f &&
             q.thresh_check > 0.f && q.thresh_check <= 1.f && q.verify <= FS_MAX_V && q.max_miss >= 1 &&
             q.max_miss <= FS_MAX_MISS && q.window <= FS_MAX_W && q.period <= FS_MAX_F &&
             (size_t)q.period > Lp + 2 * (size_t)q.window;
    }
    if (!ok) return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_fsync>(err, cfg->device, cfg->stream, [&](sdr_fsync &h) {
        const size_t C = cfg->n_channels;
        h.C = C;
        h.Lp = Lp;
        h.words.resize(cfg->n_words * Lp);
        for (size_t j = 0; j < cfg->n_words * Lp; ++j)
            h.words[j] = make_float2(cfg->words[2 * j], cfg->words[2 * j + 1]);
        h.chans.resize(C);
        h.total.assign(C, 0);
        for (size_t k = 0; k < C; ++k) {
            const size_t w = cfg->n_words == 1 ? 0 : k;
            const sdr_fsync_params_t &q = cfg->params[cfg->n_params == 1 ? 0 : k];
            h.chans[k] = FsChan{(long long)(w * Lp), (long long)h.tail_len, Ep[w], q.thresh_search, q.thresh_check,
                                q.period, q.order, q.verify, q.max_miss, q.window};
            h.tail_len += Lp + 2 * q.window;
        }
        return SDR_OK;
    });
}

extern "C" void sdr_fsync_destroy(sdr_fsync_t *h) { destroy_handle(h); }

extern "C" int sdr_fsync_reset(sdr_fsync_t *h) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    std::fill(h->total.begin(), h->total.end(), 0ull);
    h->fresh = true;  // the next call uploads the creation state (nothing carried)
    h->cur = 0;
    return SDR_OK;
}

extern "C" sdr_fsync_t *sdr_fsync_clone(const sdr_fsync_t *src, int *err) { return clone_handle<FsyncHost>(src, err); }

extern "C" int sdr_fsync_max_output(const sdr_fsync_t *h, const size_t *n_in, size_t *pay_caps, size_t *rec_caps) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_in || !pay_caps || !rec_caps) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) {
        const FsChan &c = h->chans[k];
        const unsigned long long n = n_in[k], T = h->total[k];
        if (n > FS_MAX_POS - 1 - T) return SDR_ERR_INVALID_ARG;
        if (n == 0) {
            pay_caps[k] = rec_caps[k] = 0;
            continue;
        }
        const unsigned long long mult = h->Lp >= c.W ? 1 : 2, G = c.F - c.W + 1;
        pay_caps[k] = (size_t)(mult * (n + std::min<unsigned long long>(T, h->Lp + 2 * c.W - 1)));
        rec_caps[k] = (size_t)std::min(n, 2 * ((n - 1) / G) + 2);
    }
    return SDR_OK;
}

extern "C" int sdr_fsync_get_state(sdr_fsync_t *h, size_t channel, sdr_fsync_state_t *out) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!out) return SDR_ERR_BAD_DATA_PTR;
    if (channel >= h->C) return SDR_ERR_INVALID_ARG;
    FsState st{};
    if (!h->fresh) {
        DeviceGuard g(h->dev);
        if (!g.ok) return g.status();
        SDR_CUDA_TRY(cudaMemcpyAsync(&st, (const FsState *)h->d_state.p + channel, sizeof(FsState),
                                     cudaMemcpyDeviceToHost, h->stream.s));
        SDR_CUDA_TRY(cudaStreamSynchronize(h->stream.s));
    }
    *out = sdr_fsync_state_t{st.state, st.cnt, st.pos, st.R, 0, st.consumed, st.payload};
    return SDR_OK;
}

// in: C device rows (row stride in_stride), row k of n_in[k] symbols; payload rows of out_stride, record rows of
// rec_stride (recs may be null).  Returns once the counts are on the host.
static int fs_run(sdr_fsync *h, const float2 *in, const size_t *n_in, size_t in_stride, float2 *out,
                  size_t out_stride, sdr_fsync_record_t *recs, size_t rec_stride, size_t *n_out, size_t *n_rec) {
    cudaStream_t st = h->stream.s;
    const size_t C = h->C;
    for (size_t k = 0; k < C; ++k) n_out[k] = n_rec[k] = 0;
    if (std::all_of(n_in, n_in + C, [](size_t n) { return n == 0; })) return SDR_OK;
    h->n_host.assign(n_in, n_in + C);
    h->cnt_host.resize(2 * C);
    if (h->fresh) {
        SDR_CUDA_TRY(cudaMemsetAsync(h->d_state.p, 0, C * sizeof(FsState), st));  // SEARCH from 0, nothing carried
        h->fresh = false;
    }
    long long *d_n = (long long *)h->d_n.p;
    SDR_CUDA_TRY(cudaMemcpyAsync(d_n, h->n_host.data(), C * sizeof(long long), cudaMemcpyHostToDevice, st));
    const unsigned blocks = (unsigned)((C + FS_WARPS - 1) / FS_WARPS);
    fsync_kernel<<<blocks, FS_WARPS * 32, fs_smem(h->Lp), st>>>(
        (const FsChan *)h->d_chans.p, (const float2 *)h->d_words.p, (FsState *)h->d_state.p, d_n, (int)C, (int)h->Lp,
        (float)(std::sqrt(2.0) - 1.0), (float)(1.0 / std::sqrt(2.0)), (const float2 *)h->d_tail[h->cur].p,
        (float2 *)h->d_tail[h->cur ^ 1].p, in, C > 1 ? (long long)in_stride : 0, out,
        C > 1 ? (long long)out_stride : 0, recs, C > 1 ? (long long)rec_stride : 0, d_n + C);
    count_launch();
    int rc = launch_status();
    if (rc) return rc;
    h->cur ^= 1;
    for (size_t k = 0; k < C; ++k) h->total[k] += n_in[k];
    SDR_CUDA_TRY(cudaMemcpyAsync(h->cnt_host.data(), d_n + C, 2 * C * sizeof(long long), cudaMemcpyDeviceToHost, st));
    SDR_CUDA_TRY(cudaStreamSynchronize(st));
    for (size_t k = 0; k < C; ++k) {
        n_out[k] = (size_t)h->cnt_host[k];
        n_rec[k] = (size_t)h->cnt_host[C + k];
    }
    return SDR_OK;
}

static int fs_check(const sdr_fsync *h, const float *in, const size_t *n_in, size_t in_stride, const float *out,
                    size_t out_cap, size_t out_stride, size_t *n_out, const sdr_fsync_record_t *recs, size_t rec_cap,
                    size_t rec_stride, size_t *n_rec, size_t *longest) {
    if (!h) return SDR_ERR_NULL_HANDLE;
    if (!n_out || !n_in) return SDR_ERR_BAD_DATA_PTR;
    for (size_t k = 0; k < h->C; ++k) {
        n_out[k] = 0;
        if (n_rec) n_rec[k] = 0;
    }
    *longest = *std::max_element(n_in, n_in + h->C);
    if (*longest > 0 && !in) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && in_stride < *longest) return SDR_ERR_INVALID_ARG;
    std::vector<size_t> pc(h->C), rcap(h->C);
    int rc = sdr_fsync_max_output(h, n_in, pc.data(), rcap.data());
    if (rc) return rc;
    const size_t most = *std::max_element(pc.begin(), pc.end());
    const size_t most_r = *std::max_element(rcap.begin(), rcap.end());
    if (most > out_cap || (recs && most_r > rec_cap)) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (most > 0 && !out) return SDR_ERR_BAD_DATA_PTR;
    if (h->C > 1 && ((most > 0 && out_stride < most) || (recs && most_r > 0 && rec_stride < most_r)))
        return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

extern "C" int sdr_fsync_process_dev(sdr_fsync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                     float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out,
                                     sdr_fsync_record_t *recs, size_t rec_cap, size_t rec_stride, size_t *n_rec) {
    size_t longest = 0;
    int rc = fs_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, recs, rec_cap, rec_stride,
                      n_rec, &longest);
    if (rc || longest == 0) return rc;
    if (((uintptr_t)in_c64 % 8) != 0 || ((uintptr_t)out_c64 % 8) != 0 || ((uintptr_t)recs % 8) != 0)
        return SDR_ERR_MISALIGNED;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    std::vector<size_t> nr(h->C);
    rc = fs_run(h, (const float2 *)in_c64, n_in, in_stride, (float2 *)out_c64, out_stride, recs, rec_stride, n_out,
                nr.data());
    if (!rc && n_rec) std::copy(nr.begin(), nr.end(), n_rec);
    return rc;
}

extern "C" int sdr_fsync_process(sdr_fsync_t *h, const float *in_c64, const size_t *n_in, size_t in_stride,
                                 float *out_c64, size_t out_cap, size_t out_stride, size_t *n_out,
                                 sdr_fsync_record_t *recs, size_t rec_cap, size_t rec_stride, size_t *n_rec) {
    size_t longest = 0;
    int rc = fs_check(h, in_c64, n_in, in_stride, out_c64, out_cap, out_stride, n_out, recs, rec_cap, rec_stride,
                      n_rec, &longest);
    if (rc || longest == 0) return rc;
    DeviceGuard g(h->dev);
    if (!g.ok) return g.status();
    const size_t C = h->C;
    const size_t stride = C > 1 ? in_stride : longest, ostride = C > 1 ? out_stride : out_cap,
                 rstride = C > 1 ? rec_stride : rec_cap;
    cudaStream_t st = h->stream.s;
    // rounds of up to `chunk` symbols per channel: H2D, compute (which returns the counts), D2H
    const size_t chunk = std::min(longest, std::max<size_t>(1, FS_HOST_BYTES / (C * 8)));
    const bool equal_in = std::all_of(n_in, n_in + C, [&](size_t n) { return n == longest; });
    std::vector<size_t> take(C), pc(C), rcap(C), part(C), rpart(C), done(C, 0), rdone(C, 0);
    // per-round device rows: the bounds of a full round at the largest carry
    size_t fcap = 1, rfcap = 1;
    for (size_t k = 0; k < C; ++k) {
        const FsChan &c = h->chans[k];
        const size_t mult = h->Lp >= c.W ? 1 : 2;
        fcap = std::max(fcap, mult * (chunk + h->Lp + 2 * c.W - 1));
        rfcap = std::max(rfcap, std::min(chunk, 2 * ((chunk - 1) / (c.F - c.W + 1)) + 2));
    }
    rc = h->d_in.reserve(chunk * C * 8);
    if (!rc) rc = h->d_out.reserve(fcap * C * 8);
    if (!rc && recs) rc = h->d_rec.reserve(rfcap * C * sizeof(sdr_fsync_record_t));
    if (rc) return rc;
    // one array of C rows from the device rows (cap apart) to the caller's rows (hs apart) at at[k]
    auto fetch = [&](void *dst, size_t hs, const void *src, size_t cap, size_t bytes, const std::vector<size_t> &cnt,
                     const std::vector<size_t> &at) -> int {
        for (size_t k = 0; k < C; ++k)
            if (cnt[k])
                SDR_CUDA_TRY(cudaMemcpyAsync((char *)dst + (k * hs + at[k]) * bytes, (const char *)src + k * cap * bytes,
                                             cnt[k] * bytes, cudaMemcpyDeviceToHost, st));
        return SDR_OK;
    };
    for (size_t at = 0; at < longest; at += chunk) {
        for (size_t k = 0; k < C; ++k) take[k] = n_in[k] > at ? std::min(chunk, n_in[k] - at) : 0;
        if (equal_in)
            SDR_CUDA_TRY(cudaMemcpy2DAsync(h->d_in.p, chunk * 8, in_c64 + 2 * at, stride * 8, take[0] * 8, C,
                                           cudaMemcpyHostToDevice, st));
        else
            for (size_t k = 0; k < C; ++k)
                if (take[k])
                    SDR_CUDA_TRY(cudaMemcpyAsync((float2 *)h->d_in.p + k * chunk, in_c64 + 2 * (k * stride + at),
                                                 take[k] * 8, cudaMemcpyHostToDevice, st));
        rc = fs_run(h, (const float2 *)h->d_in.p, take.data(), chunk, (float2 *)h->d_out.p, fcap,
                    recs ? (sdr_fsync_record_t *)h->d_rec.p : nullptr, rfcap, part.data(), rpart.data());
        if (rc) return rc;
        if ((rc = fetch(out_c64, ostride, h->d_out.p, fcap, 8, part, done))) return rc;
        if (recs && (rc = fetch(recs, rstride, h->d_rec.p, rfcap, sizeof(sdr_fsync_record_t), rpart, rdone)))
            return rc;
        for (size_t k = 0; k < C; ++k) {
            done[k] += part[k];
            rdone[k] += rpart[k];
        }
    }
    rc = cuda_status(cudaStreamSynchronize(st));
    if (rc) return rc;
    for (size_t k = 0; k < C; ++k) {
        n_out[k] = done[k];
        if (n_rec) n_rec[k] = rdone[k];
    }
    return SDR_OK;
}

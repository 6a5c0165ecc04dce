// fm.cu -- sdr_fm_*: the FM broadcast stereo receiver of src/main.rs:32-81 as ONE device-resident pipeline for a batch
// of stations.  Stage by stage it is the reference's chain, every intermediate stays in HBM:
//
//   u8 IQ @ rate                         RtlTcpSignal::next              rtltcp.rs:158-164
//   -> Pll(0 Hz, gain 0.035, LowPass(80 k, 0.7), Identity, LowPass(20 k, 0.7))     main.rs:41-46,49
//   -> |f| f.unwrap_or(0.0) / 75000.0                                              main.rs:49
//   -> resample_with(SincFastest, 48000 * 3)                                       main.rs:50
//   -> pilot Pll(19 kHz, gain 0.0002, LowPass(200), LowPass(20), LowPass(20)) + (mono, diff) decode   main.rs:54-71
//   -> resample(48000)   (SincBestQuality, signal/mod.rs:83; 2 channels, resample.rs:280-282)          main.rs:73
//   -> Lr(1 / 75 us) de-emphasis on mono and diff, (mono + diff, mono - diff)                         main.rs:52,75-80
//
// The `.block(0.1)` adaptors between the stages only prefetch (block.rs:148-203) and `.monitor` only prints; neither
// changes a sample.  This file is host-side composition of the library's own operators (sdr_pll_*, sdr_src_*,
// sdr_biquad_*) on one stream plus three elementwise kernels (pll.cu); it holds no arithmetic of its own.
#include <cmath>
#include <new>
#include <vector>

#include "kernels.h"

using namespace sdr;

struct FmHost {
    int dev = 0;
    size_t n_st = 0;
    float rate = 0.f, rate_mid = 0.f, rate_out = 0.f;
    float pilot_hz = 19000.0f;
    unsigned pll_flags = 0;
    double ratio1 = 0.0, ratio2 = 0.0;
};

using SrcHandle = Owned<SDR_SRC_STATE, sdr_src_delete>;

struct sdr_fm : FmHost {
    StreamRef stream;
    Owned<sdr_pll_t, sdr_pll_destroy> demod, pilot;
    std::vector<SrcHandle> src1, src2;
    Owned<sdr_biquad_t, sdr_biquad_destroy> deemph;
    DevBuf d_iq, d_c64, d_v, d_lk, d_v2, d_md, d_md2, d_out;

    int alloc(void *user_stream, const sdr_fm *);
};

// A sinc converter withholds the outputs whose right wing it has not seen yet and hands them over in a later call (or
// at the flush): at most half_len / increment = 143 output frames for ratio <= 1 (SincBestQuality).  Every per-call
// capacity carries this slack on top of ceil(n * ratio).
static const size_t kFmSlack = 256;

// the stages of one receiver, all on the handle's stream
int sdr_fm::alloc(void *user_stream, const sdr_fm *) {
    int rc = stream.init(user_stream);
    if (rc) return rc;
    void *st = (void *)stream.s;

    sdr_pll_design_t dd;  // main.rs:41-46
    dd.reference = 0.0f; dd.gain = 0.035f;
    dd.loopfilter = {SDR_BQ_LOWPASS, 80000.0f, 0.7f};
    dd.outputfilter = {SDR_BQ_IDENTITY, 0.f, 0.f};
    dd.lockfilter = {SDR_BQ_LOWPASS, 20000.0f, 0.7f};
    sdr_pll_config_t pc = {&dd, 1, n_st, rate, pll_flags, dev, st};
    demod.reset(sdr_pll_create(&pc, &rc));
    if (!demod) return rc;

    sdr_pll_design_t pd;  // main.rs:54-60
    pd.reference = pilot_hz; pd.gain = 0.0002f;
    pd.loopfilter = {SDR_BQ_LOWPASS, 200.0f, 0.7f};
    pd.outputfilter = {SDR_BQ_LOWPASS, 20.0f, 0.7f};
    pd.lockfilter = {SDR_BQ_LOWPASS, 20.0f, 0.7f};
    sdr_pll_config_t pp = {&pd, 1, n_st, rate_mid, pll_flags, dev, st};
    pilot.reset(sdr_pll_create(&pp, &rc));
    if (!pilot) return rc;

    src1.resize(n_st);
    src2.resize(n_st);
    for (size_t i = 0; i < n_st; ++i) {
        src1[i].reset(sdr_src_new_on(SDR_SRC_SINC_FASTEST, 1, dev, st, &rc));                     // main.rs:50
        if (src1[i]) src2[i].reset(sdr_src_new_on(SDR_SRC_SINC_BEST_QUALITY, 2, dev, st, &rc));  // main.rs:73
        if (!src1[i] || !src2[i]) return rc ? rc : SDR_ERR_MALLOC_FAILED;
    }
    sdr_biquad_design_t de = {SDR_BQ_LR, 1.0f / (75.0f * 0.001f * 0.001f), 0.f};  // main.rs:52
    sdr_biquad_config_t bc;
    bc.designs = &de; bc.n_designs = 1; bc.n_streams = n_st; bc.rate = rate_out;
    bc.sample_complex = 1;  // (mono, diff) frames: both parts through the same real coefficients (main.rs:74-78)
    bc.device = dev; bc.stream = st;
    deemph.reset(sdr_biquad_create(&bc, &rc));
    return deemph ? SDR_OK : rc;
}

extern "C" sdr_fm_t *sdr_fm_create(const sdr_fm_config_t *cfg, int *err) {
    if (!cfg || cfg->n_stations == 0 || cfg->n_stations > (1u << 16) || !(cfg->rate >= 144000.0f))
        return fail(err, SDR_ERR_INVALID_ARG);
    return create_handle<sdr_fm>(err, cfg->device, cfg->stream, [&](sdr_fm &f) {
        f.n_st = cfg->n_stations;
        f.rate = cfg->rate;
        f.rate_mid = 48000.0f * 3.0f;  // main.rs:50
        f.rate_out = 48000.0f;         // main.rs:73
        f.pilot_hz = cfg->pilot > 0.f ? cfg->pilot : 19000.0f;
        f.pll_flags = cfg->flags & (SDR_PLL_FAST_MATH | SDR_PLL_F64_MATH);
        // Resample::new: ratio = rate as f64 / signal.rate() as f64   (adapters/resample.rs:25)
        f.ratio1 = (double)f.rate_mid / (double)f.rate;
        f.ratio2 = (double)f.rate_out / (double)f.rate_mid;
        return SDR_OK;
    });
}

extern "C" void sdr_fm_destroy(sdr_fm_t *f) { destroy_handle(f); }

extern "C" int sdr_fm_reset(sdr_fm_t *f) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    int rc = sdr_pll_reset(f->demod.get());
    if (!rc) rc = sdr_pll_reset(f->pilot.get());
    for (size_t i = 0; i < f->n_st && !rc; ++i) {
        rc = sdr_src_reset(f->src1[i].get());
        if (!rc) rc = sdr_src_reset(f->src2[i].get());
    }
    if (!rc) rc = sdr_biquad_reset(f->deemph.get());
    return rc;
}

extern "C" float sdr_fm_output_rate(const sdr_fm_t *f) { return f ? f->rate_out : 0.f; }

extern "C" size_t sdr_fm_max_output(const sdr_fm_t *f, size_t n) {
    if (!f) return 0;
    const size_t mid = (size_t)std::ceil((double)n * f->ratio1) + kFmSlack;
    return (size_t)std::ceil((double)mid * f->ratio2) + kFmSlack;
}

// one resampler stage for every station: rows of `n_in` frames -> rows of up to `cap` frames.  All stations see the
// same counts (they depend on the call history only).  With end_of_input the converter is flushed the way the
// Resample adaptor does it (empty input => end_of_input, until nothing comes back: adapters/resample.rs:45-65).
static int fm_resample(std::vector<SrcHandle> &src, double ratio, int ch, const float *in, size_t n_in,
                       size_t in_stride, float *out, size_t cap, size_t out_stride, int end_of_input, size_t *n_out) {
    size_t gen0 = 0;
    for (size_t i = 0; i < src.size(); ++i) {
        size_t gen = 0;
        SDR_SRC_DATA d;
        d.data_in = in + i * in_stride * ch;
        d.data_out = out + i * out_stride * ch;
        d.input_frames = (long)n_in;
        d.output_frames = (long)cap;
        d.input_frames_used = d.output_frames_gen = 0;
        d.end_of_input = 0;
        d.src_ratio = ratio;
        if (n_in > 0) {
            const int rc = sdr_src_process_dev(src[i].get(), &d);
            if (rc) return rc;
            if ((size_t)d.input_frames_used != n_in) return SDR_ERR_OUTPUT_TOO_SMALL;
            gen = (size_t)d.output_frames_gen;
        }
        if (end_of_input) {
            for (;;) {
                d.data_in = in;  // not read
                d.data_out = out + (i * out_stride + gen) * ch;
                d.input_frames = 0;
                d.output_frames = (long)(cap - gen);
                d.end_of_input = 1;
                const int rc = sdr_src_process_dev(src[i].get(), &d);
                if (rc) return rc;
                if (d.output_frames_gen == 0) break;
                gen += (size_t)d.output_frames_gen;
                if (gen >= cap) return SDR_ERR_OUTPUT_TOO_SMALL;
            }
        }
        if (i == 0) gen0 = gen;
        else if (gen != gen0) return SDR_ERR_BAD_STATE;
    }
    *n_out = gen0;
    return SDR_OK;
}

static int fm_run(sdr_fm *f, const uint8_t *d_iq, size_t n, size_t in_stride, float *d_out, size_t out_cap,
                  size_t out_stride, size_t *n_out, int end_of_input) {
    const size_t S = f->n_st;
    cudaStream_t st = f->stream.s;
    // reject a short output buffer BEFORE any stage consumes the block: the PLLs and converters advance their state
    // as they run, so a late SDR_ERR_OUTPUT_TOO_SMALL would drop samples and leave a handle that cannot be retried
    if (out_cap < sdr_fm_max_output(f, n)) return SDR_ERR_OUTPUT_TOO_SMALL;
    const size_t cap2 = (size_t)std::ceil((double)n * f->ratio1) + kFmSlack;
    const size_t cap3 = (size_t)std::ceil((double)cap2 * f->ratio2) + kFmSlack;
    const size_t nc = (n + 1) & ~(size_t)1;  // c64 row pitch: keeps every row 16-byte aligned for the unpack kernel
    int rc = f->d_c64.reserve(S * nc * 8 + 16);
    if (!rc) rc = f->d_v.reserve(S * n * 4 + 16);
    if (!rc) rc = f->d_lk.reserve(S * n + 16);
    if (!rc) rc = f->d_v2.reserve(S * cap2 * 4);
    if (!rc) rc = f->d_md.reserve(S * cap2 * 8);
    if (!rc) rc = f->d_md2.reserve(S * cap3 * 8);
    if (rc) return rc;
    float *c64 = (float *)f->d_c64.p, *v = (float *)f->d_v.p, *v2 = (float *)f->d_v2.p, *md = (float *)f->d_md.p,
          *md2 = (float *)f->d_md2.p;
    uint8_t *lk = (uint8_t *)f->d_lk.p;
    if (n > 0) {
        for (size_t i = 0; i < S && !rc; ++i)  // rows may be padded on the caller's side
            rc = sdr_unpack_u8iq_dev(d_iq + i * in_stride, n, c64 + 2 * i * nc, f->dev, (void *)st);
        if (!rc) rc = sdr_pll_process_dev(f->demod.get(), c64, n, nc, v, lk, n);
        if (!rc) rc = fm_demod_map_launch(v, lk, v, (long long)(S * n), st);
        if (rc) return rc;
    }
    size_t n2 = 0, n3 = 0;
    rc = fm_resample(f->src1, f->ratio1, 1, v, n, n, v2, cap2, cap2, end_of_input, &n2);
    if (rc) return rc;
    if (n2 > 0) {
        rc = sdr_pll_stereo_decode_dev(f->pilot.get(), v2, n2, cap2, md, cap2);
        if (rc) return rc;
    }
    rc = fm_resample(f->src2, f->ratio2, 2, md, n2, cap2, md2, cap3, cap3, end_of_input, &n3);
    if (rc) return rc;
    if (n3 > out_cap) return SDR_ERR_OUTPUT_TOO_SMALL;
    if (n3 > 0) {
        rc = sdr_biquad_process_dev(f->deemph.get(), md2, n3, cap3, md2, cap3);
        if (!rc) rc = fm_matrix_launch(md2, (long long)cap3, d_out, (long long)out_stride, (int)S, (long long)n3, st);
        if (rc) return rc;
    }
    *n_out = n3;
    return SDR_OK;
}

extern "C" int sdr_fm_process_dev(sdr_fm_t *f, const uint8_t *iq, size_t n, size_t in_stride, float *out,
                                  size_t out_cap, size_t out_stride, size_t *n_out, int end_of_input) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    if (!n_out || (n > 0 && !iq) || !out) return SDR_ERR_BAD_DATA_PTR;
    if (f->n_st == 1) { in_stride = 2 * n; out_stride = out_cap; }
    if (in_stride < 2 * n || out_stride < out_cap) return SDR_ERR_INVALID_ARG;
    if (f->n_st > 1 && (in_stride & 15)) return SDR_ERR_MISALIGNED;  // rows feed a 16-byte vectorised unpack
    DeviceGuard g(f->dev);
    if (!g.ok) return g.status();
    return fm_run(f, iq, n, in_stride, out, out_cap, out_stride, n_out, end_of_input);
}

extern "C" int sdr_fm_process(sdr_fm_t *f, const uint8_t *iq, size_t n, size_t in_stride, float *out, size_t out_cap,
                              size_t out_stride, size_t *n_out, int end_of_input) {
    if (!f) return SDR_ERR_NULL_HANDLE;
    if (!n_out || (n > 0 && !iq) || !out) return SDR_ERR_BAD_DATA_PTR;
    if (f->n_st == 1) { in_stride = 2 * n; out_stride = out_cap; }
    if (in_stride < 2 * n || out_stride < out_cap) return SDR_ERR_INVALID_ARG;
    DeviceGuard g(f->dev);
    if (!g.ok) return g.status();
    const size_t S = f->n_st;
    cudaStream_t st = f->stream.s;
    const size_t row = (2 * n + 15) & ~(size_t)15;  // 16-byte aligned rows for the unpack kernel
    int rc = f->d_iq.reserve(S * row + 16);
    if (!rc) rc = f->d_out.reserve(S * out_cap * 8 + 16);
    if (rc) return rc;
    if (n > 0) {
        SDR_CUDA_TRY(cudaMemcpy2DAsync(f->d_iq.p, row, iq, in_stride, 2 * n, S, cudaMemcpyHostToDevice, st));
    }
    rc = fm_run(f, (const uint8_t *)f->d_iq.p, n, row, (float *)f->d_out.p, out_cap, out_cap, n_out, end_of_input);
    if (rc) return rc;
    if (*n_out > 0) {
        SDR_CUDA_TRY(cudaMemcpy2DAsync(out, out_stride * 8, f->d_out.p, out_cap * 8, *n_out * 8, S,
                                       cudaMemcpyDeviceToHost, st));
    }
    return cuda_status(cudaStreamSynchronize(st));
}

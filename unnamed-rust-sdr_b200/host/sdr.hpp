// sdr.hpp -- C++ host-side mirror of the reference crate's public API for the hot path, sitting on
// the C ABI of include/sdr_b200.h.  (The reference is Rust; this image has no Rust toolchain, so the
// host side above the boundary is written in C++ -- same names, argument meaning and error behaviour.
// The Rust binding a maintainer would add is in ../rust/ and INTEGRATION.md.)
//
//   reference                                          here
//   ------------------------------------------------   -------------------------------------------
//   num::Complex<f32>                                  sdr::Complex
//   trait Signal {next, rate, + combinators}           sdr::signal::Signal<Sample> (block pull) with the same
//     (src/signal/mod.rs:13-123)                         combinators: block decimate filter map resample
//                                                        resample_with skip take iter
//   signal::from_iter (sources.rs:31-36)               sdr::signal::from_iter(rate, vector)
//   rtltcp::RtlTcpSignal (rtltcp.rs:151-168)           sdr::signal::from_u8iq(rate, bytes)
//   filter::Fir<C,A>, FilterDesign for Vec<C>          sdr::filter::Fir<C,A>  (+ block process(), mirroring
//     (src/filter/fir.rs)                                SampleRate::process, since a per-sample GPU call is absurd)
//   filter::BiquadD, Biquad, Identity, PllDesign, Pll  sdr::filter::BiquadD, Biquad<A>, Identity, PllDesign, Pll
//   resample::SampleRate<A>, ConverterType, Error      sdr::resample::SampleRate<A>, ConverterType, Error
//     (src/resample.rs)
//   fft::fft, fft::rfft (src/fft.rs)                   sdr::fft::fft, sdr::fft::rfft
//
// Errors: the reference returns Result and its adaptors unwrap() (panic); here constructors / process
// throw sdr::Error / sdr::resample::Error, which is the same "abort the pipeline" behaviour.
#pragma once
#include <algorithm>
#include <complex>
#include <cstdint>
#include <deque>
#include <functional>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/sdr_b200.h"

namespace sdr {

using Complex = std::complex<float>;

struct Error : std::runtime_error {
    int code;
    Error(int c, const char *what) : std::runtime_error(std::string(what) + ": " + sdr_strerror(c)), code(c) {}
};
inline void check(int rc, const char *what) {
    if (rc != SDR_OK) throw Error(rc, what);
}

// Owner of one ABI handle for the mirror classes: a move transfers it, a copy clones it (its stream state included)
// and destruction destroys it.
template <class T, void (*Destroy)(T *), T *(*Clone)(const T *, int *)>
class Handle {
  protected:
    T *h_ = nullptr;
    Handle() = default;
    Handle(Handle &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    Handle(const Handle &o) {
        int err = 0;
        h_ = Clone(o.h_, &err);
        if (!h_) throw Error(err, "clone");
    }
    Handle &operator=(const Handle &) = delete;
    ~Handle() { Destroy(h_); }
};

template <class A> struct SampleTraits;
template <> struct SampleTraits<float> { static constexpr int fmt = SDR_FMT_F32; static constexpr int channels = 1; };
template <> struct SampleTraits<Complex> { static constexpr int fmt = SDR_FMT_C64; static constexpr int channels = 2; };
template <class A, class B> struct SampleTraits<std::pair<A, B>> {  // resample.rs:280-282
    static constexpr int channels = SampleTraits<A>::channels + SampleTraits<B>::channels;
};

// =========================================================================================
namespace resample {

enum class ConverterType {  // resample.rs:112-119
    SincBestQuality = SDR_SRC_SINC_BEST_QUALITY,
    SincMediumQuality = SDR_SRC_SINC_MEDIUM_QUALITY,
    SincFastest = SDR_SRC_SINC_FASTEST,
    ZeroOrderHold = SDR_SRC_ZERO_ORDER_HOLD,
    Linear = SDR_SRC_LINEAR,
};
inline const char *name(ConverterType t) { return sdr_src_get_name((int)t); }
inline const char *description(ConverterType t) { return sdr_src_get_description((int)t); }
inline const char *version() { return sdr_src_get_version(); }

struct Error : std::runtime_error {  // resample.rs:151-270
    int code;
    explicit Error(int c) : std::runtime_error(sdr_src_strerror(c) ? sdr_src_strerror(c) : "Unknown"), code(c) {}
};

// SampleRate<A>: A is memory-identical to [f32; channels] (resample.rs:27-30)
template <class A>
class SampleRate {
    SDR_SRC_STATE *state_ = nullptr;
    explicit SampleRate(SDR_SRC_STATE *s) : state_(s) {}

  public:
    explicit SampleRate(ConverterType typ) {  // SampleRate::new (resample.rs:33-44)
        int err = 0;
        state_ = sdr_src_new((int)typ, SampleTraits<A>::channels, &err);
        if (!state_ || err) throw Error(err);
    }
    SampleRate(SampleRate &&o) noexcept : state_(o.state_) { o.state_ = nullptr; }
    SampleRate &operator=(SampleRate &&o) noexcept { std::swap(state_, o.state_); return *this; }
    SampleRate(const SampleRate &o) : state_(nullptr) { *this = o.try_clone(); }  // impl Clone (resample.rs:17-21)
    ~SampleRate() { if (state_) state_ = sdr_src_delete(state_); }              // Drop (resample.rs:101-110)

    // process(ratio, &input, &mut output) -> input_frames_used; output.len = output_frames_gen;
    // output_frames = output.capacity(); end_of_input = input.is_empty()   (resample.rs:46-67)
    size_t process(double ratio, const std::vector<A> &input, std::vector<A> &output) {
        const size_t cap = output.capacity();
        output.resize(cap);
        SDR_SRC_DATA cmd;
        cmd.data_in = reinterpret_cast<const float *>(input.data());
        cmd.data_out = reinterpret_cast<float *>(output.data());
        cmd.input_frames = (long)input.size();
        cmd.output_frames = (long)cap;
        cmd.input_frames_used = 0;
        cmd.output_frames_gen = 0;
        cmd.end_of_input = input.empty() ? 1 : 0;
        cmd.src_ratio = ratio;
        const int rc = sdr_src_process(state_, &cmd);
        if (rc) { output.resize(0); throw Error(rc); }
        output.resize((size_t)cmd.output_frames_gen);
        return (size_t)cmd.input_frames_used;
    }
    void reset() { int rc = sdr_src_reset(state_); if (rc) throw Error(rc); }
    SampleRate try_clone() const {
        int err = 0;
        SDR_SRC_STATE *s = sdr_src_clone(state_, &err);
        if (!s || err) throw Error(err);
        return SampleRate(s);
    }
    size_t channels() const { return (size_t)sdr_src_get_channels(state_); }
    void set_ratio(double r) { int rc = sdr_src_set_ratio(state_, r); if (rc) throw Error(rc); }
};

}  // namespace resample

// =========================================================================================
namespace filter {

// Fir<C,A> (src/filter/fir.rs:7-33).  C in {float, Complex}; A in {float, Complex}; also usable with
// input_u8iq = true, where the samples arrive as rtl_tcp bytes and are unpacked on the GPU.
template <class C, class A>
class Fir : public Handle<sdr_fir_t, sdr_fir_destroy, sdr_fir_clone> {
    std::vector<C> coef_;

  public:
    explicit Fir(std::vector<C> coef, size_t decimation = 1, bool input_u8iq = false, unsigned flags = 0)
        : coef_(std::move(coef)) {
        static_assert(!(std::is_same<C, Complex>::value && std::is_same<A, float>::value),
                      "f32 * Complex<f32> is not a Convolve impl in the reference");
        sdr_fir_config_t cfg{};
        cfg.taps = reinterpret_cast<const float *>(coef_.data());
        cfg.n_taps = coef_.size();
        cfg.taps_complex = std::is_same<C, Complex>::value;
        cfg.input_format = input_u8iq ? SDR_FMT_U8IQ : SampleTraits<A>::fmt;
        cfg.decimation = decimation;
        cfg.n_channels = 1;
        cfg.flags = flags;
        cfg.device = 0;
        cfg.stream = nullptr;
        int err = 0;
        h_ = sdr_fir_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Fir::new");
    }

    // block form of Filter::apply: out gets one element per kept input (all of them when decimation == 1)
    void process(const void *in, size_t n_in, std::vector<A> &out) {
        const size_t n_out = sdr_fir_output_count(h_, n_in);
        out.resize(n_out);
        size_t used = 0, got = 0;
        check(sdr_fir_process(h_, in, n_in, n_in, out.data(), n_out, n_out, &used, &got), "Fir::process");
        out.resize(got);
    }
    A apply(A value) {  // Filter::apply (filter/mod.rs:23-26); one launch per sample: correct, not fast
        std::vector<A> o;
        process(&value, 1, o);
        return o.empty() ? A() : o[0];
    }
    void reset() { check(sdr_fir_reset(h_), "Fir::reset"); }
    const std::vector<C> &coef() const { return coef_; }
};

// Polyphase filter bank behind sdr_pfb_*: channel k is Fir<Complex, Complex>(h[n] e^{+2 pi i k n / M}) followed by
// Decimate(D), for k = 0..M-1, computed in one pass over the input.  flags: SDR_PFB_SHIFT, SDR_PFB_CHANNEL_MAJOR.
class Pfb : public Handle<sdr_pfb_t, sdr_pfb_destroy, sdr_pfb_clone> {
    size_t m_ = 0;
    bool cmajor_ = false;

  public:
    Pfb(const std::vector<float> &prototype, size_t n_channels, size_t decimation, bool input_u8iq = false,
        unsigned flags = 0)
        : m_(n_channels), cmajor_((flags & SDR_PFB_CHANNEL_MAJOR) != 0) {
        sdr_pfb_config_t cfg{};
        cfg.taps = prototype.data();
        cfg.n_taps = prototype.size();
        cfg.n_channels = n_channels;
        cfg.decimation = decimation;
        cfg.input_format = input_u8iq ? SDR_FMT_U8IQ : SDR_FMT_C64;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_pfb_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Pfb::new");
    }
    size_t channels() const { return m_; }
    size_t output_count(size_t n_in) const { return sdr_pfb_output_count(h_, n_in); }
    // in: n samples (Complex, or 2n bytes when constructed with input_u8iq).  out: frames x M (or M x frames when
    // channel-major), replaced.  Returns the number of frames.
    size_t process(const void *in, size_t n, std::vector<Complex> &out) {
        const size_t nf = output_count(n);
        out.resize((nf ? nf : 1) * m_);
        size_t got = 0;
        check(sdr_pfb_process(h_, in, n, reinterpret_cast<float *>(out.data()), nf, cmajor_ ? nf : m_, &got),
              "Pfb::process");
        out.resize(got * m_);
        return got;
    }
    void reset() { check(sdr_pfb_reset(h_), "Pfb::reset"); }
};

// Polyphase synthesis bank behind sdr_pfs_*, the inverse of Pfb: channel k is zero-stuffed by D (sample m at index
// (m+1) D - 1), filtered by Fir<Complex, Complex>(f[n] e^{+2 pi i k n / M}) and summed over k; n frames give n D
// samples.  flags: SDR_PFS_SHIFT, SDR_PFS_CHANNEL_MAJOR take the layouts Pfb writes with the matching flags.
class Pfs : public Handle<sdr_pfs_t, sdr_pfs_destroy, sdr_pfs_clone> {
    size_t m_ = 0;
    bool cmajor_ = false;

  public:
    Pfs(const std::vector<float> &prototype, size_t n_channels, size_t interpolation, unsigned flags = 0)
        : m_(n_channels), cmajor_((flags & SDR_PFS_CHANNEL_MAJOR) != 0) {
        sdr_pfs_config_t cfg{};
        cfg.taps = prototype.data();
        cfg.n_taps = prototype.size();
        cfg.n_channels = n_channels;
        cfg.interpolation = interpolation;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_pfs_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Pfs::new");
    }
    size_t channels() const { return m_; }
    size_t output_count(size_t n_frames) const { return sdr_pfs_output_count(h_, n_frames); }
    // in: n_frames frames of M (or M rows of n_frames when channel-major).  out: n_frames * D samples, replaced.
    size_t process(const Complex *in, size_t n_frames, std::vector<Complex> &out) {
        const size_t n = output_count(n_frames);
        out.resize(n ? n : 1);
        size_t got = 0;
        check(sdr_pfs_process(h_, reinterpret_cast<const float *>(in), n_frames, cmajor_ ? n_frames : m_,
                              reinterpret_cast<float *>(out.data()), n, &got),
              "Pfs::process");
        out.resize(got);
        return got;
    }
    void reset() { check(sdr_pfs_reset(h_), "Pfs::reset"); }
};

// Down-converter bank behind sdr_ddc_*: channel k is a tee'd copy of the stream mixed down by a 64-bit NCO
// (sdr_ddc_phase_increment(freq[k], rate)), Fir<Complex, f32>(h_k) and Decimate(D), computed in one pass over the input.
// taps: one row of L (shared) or channels rows of L.  Output: channels rows of outputs (channel-major).
class Ddc : public Handle<sdr_ddc_t, sdr_ddc_destroy, sdr_ddc_clone> {
    size_t c_ = 0;

  public:
    Ddc(const std::vector<float> &taps, size_t n_taps, const std::vector<double> &freqs, double rate, size_t decimation,
        bool input_u8iq = true, uint64_t first_sample = 0, unsigned flags = 0)
        : c_(freqs.size()) {
        std::vector<uint64_t> inc(freqs.size());
        for (size_t k = 0; k < freqs.size(); ++k) inc[k] = sdr_ddc_phase_increment(freqs[k], rate);
        sdr_ddc_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phase_inc = inc.data();
        cfg.n_channels = freqs.size();
        cfg.decimation = decimation;
        cfg.first_sample = first_sample;
        cfg.input_format = input_u8iq ? SDR_FMT_U8IQ : SDR_FMT_C64;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_ddc_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Ddc::new");
    }
    size_t channels() const { return c_; }
    size_t output_count(size_t n_in) const { return sdr_ddc_output_count(h_, n_in); }
    int last_path() const { return sdr_ddc_last_path(h_); }
    // in: n samples (Complex, or 2n rtl_tcp bytes when constructed with input_u8iq).  out: channels x outputs,
    // replaced.  Returns the outputs per channel.
    size_t process(const void *in, size_t n, std::vector<Complex> &out) {
        const size_t nf = output_count(n);
        out.resize((nf ? nf : 1) * c_);
        size_t got = 0;
        check(sdr_ddc_process(h_, in, n, reinterpret_cast<float *>(out.data()), nf, nf ? nf : 1, &got), "Ddc::process");
        out.resize(got * c_);
        return got;
    }
    void reset() { check(sdr_ddc_reset(h_), "Ddc::reset"); }
};

// Up-converter bank behind sdr_duc_*, the transpose of Ddc: channel k is zero-stuffed by I (sample m at index
// (m+1) I - 1), filtered by Fir<f32, Complex>(h_k), mixed up by a 64-bit NCO (sdr_ddc_phase_increment(freq[k], rate))
// and the channels are summed.  taps: one row of L (shared) or channels rows of L.  Input: channels rows of frames
// (channel-major, as Ddc writes them); n frames give n I samples.
class Duc : public Handle<sdr_duc_t, sdr_duc_destroy, sdr_duc_clone> {
    size_t c_ = 0;

  public:
    Duc(const std::vector<float> &taps, size_t n_taps, const std::vector<double> &freqs, double rate,
        size_t interpolation, uint64_t first_sample = 0)
        : c_(freqs.size()) {
        std::vector<uint64_t> inc(freqs.size());
        for (size_t k = 0; k < freqs.size(); ++k) inc[k] = sdr_ddc_phase_increment(freqs[k], rate);
        sdr_duc_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phase_inc = inc.data();
        cfg.n_channels = freqs.size();
        cfg.interpolation = interpolation;
        cfg.first_sample = first_sample;
        int err = 0;
        h_ = sdr_duc_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Duc::new");
    }
    size_t channels() const { return c_; }
    size_t output_count(size_t n_frames) const { return sdr_duc_output_count(h_, n_frames); }
    // in: channels rows of n_frames, row stride in_stride (>= n_frames).  out: n_frames * I samples, replaced.
    size_t process(const Complex *in, size_t n_frames, size_t in_stride, std::vector<Complex> &out) {
        const size_t n = output_count(n_frames);
        out.resize(n ? n : 1);
        size_t got = 0;
        check(sdr_duc_process(h_, reinterpret_cast<const float *>(in), n_frames, in_stride,
                              reinterpret_cast<float *>(out.data()), n, &got),
              "Duc::process");
        out.resize(got);
        return got;
    }
    void reset() { check(sdr_duc_reset(h_), "Duc::reset"); }
};

// Fast-convolution channel bank (sdr_fcfb): Ddc's channels with one decimation per channel, computed by overlap-save.
// Outputs are released per block of P inputs (sdr_fcfb_geometry); feed N zeros to drain a finite stream.
class Fcfb : public Handle<sdr_fcfb_t, sdr_fcfb_destroy, sdr_fcfb_clone> {
    size_t c_ = 0;

  public:
    Fcfb(const std::vector<float> &taps, size_t n_taps, const std::vector<double> &freqs, double rate,
         const std::vector<size_t> &decimation, bool input_u8iq = true, uint64_t first_sample = 0)
        : c_(freqs.size()) {
        std::vector<uint64_t> inc(freqs.size());
        for (size_t k = 0; k < freqs.size(); ++k) inc[k] = sdr_ddc_phase_increment(freqs[k], rate);
        if (decimation.size() != freqs.size()) throw sdr::Error(SDR_ERR_INVALID_ARG, "Fcfb::new");
        sdr_fcfb_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phase_inc = inc.data();
        cfg.decimation = decimation.data();
        cfg.n_channels = freqs.size();
        cfg.first_sample = first_sample;
        cfg.input_format = input_u8iq ? SDR_FMT_U8IQ : SDR_FMT_C64;
        int err = 0;
        h_ = sdr_fcfb_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Fcfb::new");
    }
    size_t channels() const { return c_; }
    std::vector<size_t> output_count(size_t n_in) const {
        std::vector<size_t> cnt(c_);
        check(sdr_fcfb_output_count(h_, n_in, cnt.data()), "Fcfb::output_count");
        return cnt;
    }
    // in: n samples (Complex, or 2n rtl_tcp bytes when constructed with input_u8iq).  out: one vector per channel, replaced.
    void process(const void *in, size_t n, std::vector<std::vector<Complex>> &out) {
        const std::vector<size_t> cnt = output_count(n);
        const size_t cap = std::max<size_t>(1, *std::max_element(cnt.begin(), cnt.end()));
        std::vector<Complex> rows(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_fcfb_process(h_, in, n, reinterpret_cast<float *>(rows.data()), cap, cap, got.data()), "Fcfb::process");
        out.assign(c_, {});
        for (size_t k = 0; k < c_; ++k) out[k].assign(rows.begin() + k * cap, rows.begin() + k * cap + got[k]);
    }
    void reset() { check(sdr_fcfb_reset(h_), "Fcfb::reset"); }
};

// Fast-convolution synthesis bank (sdr_fcsb), the inverse of Fcfb: Duc's channels with one interpolation per channel,
// computed by overlap-save.  A call advances by n_time output positions (a multiple of lcm(I_k); row k holds
// n_time / I_k frames) and returns the outputs of the blocks it completes; feed zero frames covering N positions to
// drain a finite stream.
class Fcsb : public Handle<sdr_fcsb_t, sdr_fcsb_destroy, sdr_fcsb_clone> {
    size_t c_ = 0;

  public:
    Fcsb(const std::vector<float> &taps, size_t n_taps, const std::vector<double> &freqs, double rate,
         const std::vector<size_t> &interpolation, uint64_t first_sample = 0)
        : c_(freqs.size()) {
        std::vector<uint64_t> inc(freqs.size());
        for (size_t k = 0; k < freqs.size(); ++k) inc[k] = sdr_ddc_phase_increment(freqs[k], rate);
        if (interpolation.size() != freqs.size()) throw sdr::Error(SDR_ERR_INVALID_ARG, "Fcsb::new");
        sdr_fcsb_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phase_inc = inc.data();
        cfg.interpolation = interpolation.data();
        cfg.n_channels = freqs.size();
        cfg.first_sample = first_sample;
        int err = 0;
        h_ = sdr_fcsb_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Fcsb::new");
    }
    size_t channels() const { return c_; }
    size_t output_count(size_t n_time) const { return sdr_fcsb_output_count(h_, n_time); }
    // in: channels rows, row k = n_time / I_k frames, row stride in_stride (>= the longest row).  out: replaced.
    size_t process(const Complex *in, size_t n_time, size_t in_stride, std::vector<Complex> &out) {
        const size_t n = output_count(n_time);
        out.resize(n ? n : 1);
        size_t got = 0;
        check(sdr_fcsb_process(h_, reinterpret_cast<const float *>(in), n_time, in_stride,
                               reinterpret_cast<float *>(out.data()), n, &got),
              "Fcsb::process");
        out.resize(got);
        return got;
    }
    void reset() { check(sdr_fcsb_reset(h_), "Fcsb::reset"); }
};

// Rational resampler bank (sdr_rrb): channel k zero-stuffed by I_k, filtered by its real taps and decimated by D_k
// (upfirdn).  After n frames a channel has released floor(n I_k / D_k) outputs; there is no scale (taps carry I_k).
class Rrb : public Handle<sdr_rrb_t, sdr_rrb_destroy, sdr_rrb_clone> {
    size_t c_ = 0;

  public:
    Rrb(const std::vector<float> &taps, size_t n_taps, const std::vector<size_t> &interpolation,
        const std::vector<size_t> &decimation)
        : c_(interpolation.size()) {
        if (decimation.size() != interpolation.size()) throw sdr::Error(SDR_ERR_INVALID_ARG, "Rrb::new");
        sdr_rrb_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.interpolation = interpolation.data();
        cfg.decimation = decimation.data();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_rrb_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Rrb::new");
    }
    size_t channels() const { return c_; }
    std::vector<size_t> output_count(const std::vector<size_t> &n_in) const {
        std::vector<size_t> cnt(c_);
        check(sdr_rrb_output_count(h_, n_in.data(), cnt.data()), "Rrb::output_count");
        return cnt;
    }
    // in: channels rows, row k of n_in[k] frames at row stride in_stride (>= the longest row).  out: one vector per
    // channel, replaced.
    void process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride,
                 std::vector<std::vector<Complex>> &out) {
        const std::vector<size_t> cnt = output_count(n_in);
        const size_t cap = std::max<size_t>(1, *std::max_element(cnt.begin(), cnt.end()));
        std::vector<Complex> rows(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_rrb_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                              reinterpret_cast<float *>(rows.data()), cap, cap, got.data()),
              "Rrb::process");
        out.assign(c_, {});
        for (size_t k = 0; k < c_; ++k) out[k].assign(rows.begin() + k * cap, rows.begin() + k * cap + got[k]);
    }
    void reset() { check(sdr_rrb_reset(h_), "Rrb::reset"); }
};

// Arbitrary-ratio resampler bank (sdr_arb): channel k resampled by its own step (input frames per output, exact in
// units of 2^-64) with real taps designed at P times the input rate, interpolated between adjacent phases.  After n
// frames a channel has released #{r : tau(r) < n} outputs; there is no scale (unit gain needs sum h = P).
class Arb : public Handle<sdr_arb_t, sdr_arb_destroy, sdr_arb_clone> {
    size_t c_ = 0;

  public:
    // rate_in / rate_out to the nearest 2^-64
    static sdr_arb_time_t step(double rate_in, double rate_out) {
        sdr_arb_time_t t{};
        check(sdr_arb_step(rate_in, rate_out, &t), "Arb::step");
        return t;
    }
    // first: empty (all 0) or one position per channel
    Arb(const std::vector<float> &taps, size_t n_taps, size_t phases, const std::vector<sdr_arb_time_t> &steps,
        const std::vector<sdr_arb_time_t> &first = {})
        : c_(steps.size()) {
        if (!first.empty() && first.size() != steps.size()) throw sdr::Error(SDR_ERR_INVALID_ARG, "Arb::new");
        sdr_arb_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phases = phases;
        cfg.step = steps.data();
        cfg.first = first.empty() ? nullptr : first.data();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_arb_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Arb::new");
    }
    size_t channels() const { return c_; }
    void set_steps(const std::vector<sdr_arb_time_t> &steps) {
        if (steps.size() != c_) throw sdr::Error(SDR_ERR_INVALID_ARG, "Arb::set_steps");
        check(sdr_arb_set_steps(h_, steps.data()), "Arb::set_steps");
    }
    std::vector<size_t> output_count(const std::vector<size_t> &n_in) const {
        std::vector<size_t> cnt(c_);
        check(sdr_arb_output_count(h_, n_in.data(), cnt.data()), "Arb::output_count");
        return cnt;
    }
    // in: channels rows, row k of n_in[k] frames at row stride in_stride (>= the longest row).  out: one vector per
    // channel, replaced.
    void process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride,
                 std::vector<std::vector<Complex>> &out) {
        const std::vector<size_t> cnt = output_count(n_in);
        const size_t cap = std::max<size_t>(1, *std::max_element(cnt.begin(), cnt.end()));
        std::vector<Complex> rows(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_arb_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                              reinterpret_cast<float *>(rows.data()), cap, cap, got.data()),
              "Arb::process");
        out.assign(c_, {});
        for (size_t k = 0; k < c_; ++k) out[k].assign(rows.begin() + k * cap, rows.begin() + k * cap + got[k]);
    }
    void reset() { check(sdr_arb_reset(h_), "Arb::reset"); }
};

// Symbol timing recovery bank (sdr_tsync): a Gardner loop per channel steering sdr_arb's interpolator on the exact
// 64.64 time base.  Channel k: matched filter taps at P times the input rate, a nominal period (Arb::step(rate,
// symbol_rate)), a first position and loop parameters {kp, ki, err_max, max_dev}; each call returns the released symbols
// with their exact positions and detector outputs.  Counts come from the device, so every call synchronises.
class Tsync : public Handle<sdr_tsync_t, sdr_tsync_destroy, sdr_tsync_clone> {
    size_t c_ = 0;

  public:
    struct Out {
        std::vector<std::vector<Complex>> sym;
        std::vector<std::vector<sdr_arb_time_t>> pos;
        std::vector<std::vector<float>> err;
    };
    // kp, ki in frames per unit of detector output for a noise bandwidth bn_t, damping zeta and detector slope ted_gain
    static std::pair<float, float> loop_design(double bn_t, double zeta, double ted_gain, double period_frames) {
        float kp = 0, ki = 0;
        check(sdr_tsync_loop_design(bn_t, zeta, ted_gain, period_frames, &kp, &ki), "Tsync::loop_design");
        return {kp, ki};
    }
    // loops: one (shared) or one per channel; first: empty (all 0) or one position per channel
    Tsync(const std::vector<float> &taps, size_t n_taps, size_t phases, const std::vector<sdr_arb_time_t> &periods,
          const std::vector<sdr_tsync_loop_t> &loops, const std::vector<sdr_arb_time_t> &first = {})
        : c_(periods.size()) {
        if (!first.empty() && first.size() != periods.size()) throw sdr::Error(SDR_ERR_INVALID_ARG, "Tsync::new");
        sdr_tsync_config_t cfg{};
        cfg.taps = taps.data();
        cfg.n_taps = n_taps;
        cfg.n_tap_sets = n_taps ? taps.size() / n_taps : 0;
        cfg.phases = phases;
        cfg.period = periods.data();
        cfg.first = first.empty() ? nullptr : first.data();
        cfg.loops = loops.data();
        cfg.n_loops = loops.size();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_tsync_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Tsync::new");
    }
    size_t channels() const { return c_; }
    std::vector<size_t> max_output(const std::vector<size_t> &n_in) const {
        std::vector<size_t> cap(c_);
        check(sdr_tsync_max_output(h_, n_in.data(), cap.data()), "Tsync::max_output");
        return cap;
    }
    // next unreleased position and v (units of 2^-40 frames) of one channel
    std::pair<sdr_arb_time_t, int64_t> state(size_t k) {
        sdr_arb_time_t t{};
        int64_t v = 0;
        check(sdr_tsync_get_state(h_, k, &t, &v), "Tsync::state");
        return {t, v};
    }
    // in: channels rows, row k of n_in[k] frames at row stride in_stride (>= the longest row)
    Out process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride) {
        const std::vector<size_t> caps = max_output(n_in);
        const size_t cap = std::max<size_t>(1, *std::max_element(caps.begin(), caps.end()));
        std::vector<Complex> sym(cap * c_);
        std::vector<sdr_arb_time_t> pos(cap * c_);
        std::vector<float> err(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_tsync_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                                reinterpret_cast<float *>(sym.data()), pos.data(), err.data(), cap, cap, got.data()),
              "Tsync::process");
        Out o;
        o.sym.resize(c_);
        o.pos.resize(c_);
        o.err.resize(c_);
        for (size_t k = 0; k < c_; ++k) {
            o.sym[k].assign(sym.begin() + k * cap, sym.begin() + k * cap + got[k]);
            o.pos[k].assign(pos.begin() + k * cap, pos.begin() + k * cap + got[k]);
            o.err[k].assign(err.begin() + k * cap, err.begin() + k * cap + got[k]);
        }
        return o;
    }
    void reset() { check(sdr_tsync_reset(h_), "Tsync::reset"); }
};

// Carrier recovery bank (sdr_csync): a decision-directed Costas loop per channel on an exact 64-bit phase.  Channel k:
// loop parameters {order, kp, ki, err_max, max_freq} (kp, ki from Tsync::loop_design(bn_t, zeta, K_d, 1 / (2 pi))), a
// first phase (2^-64 turn) and frequency (2^-40 turn per symbol); each call returns one derotated symbol per input
// symbol with its phase and detector output.
class Csync : public Handle<sdr_csync_t, sdr_csync_destroy, sdr_csync_clone> {
    size_t c_ = 0;

  public:
    struct Out {
        std::vector<std::vector<Complex>> sym;
        std::vector<std::vector<uint64_t>> phase;
        std::vector<std::vector<float>> err;
    };
    // loops: one (shared) or one per channel; phase, freq: empty (all 0) or one per channel
    Csync(size_t channels, const std::vector<sdr_csync_loop_t> &loops, const std::vector<uint64_t> &phase = {},
          const std::vector<int64_t> &freq = {})
        : c_(channels) {
        if ((!phase.empty() && phase.size() != channels) || (!freq.empty() && freq.size() != channels))
            throw sdr::Error(SDR_ERR_INVALID_ARG, "Csync::new");
        sdr_csync_config_t cfg{};
        cfg.loops = loops.data();
        cfg.n_loops = loops.size();
        cfg.phase = phase.empty() ? nullptr : phase.data();
        cfg.freq = freq.empty() ? nullptr : freq.data();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_csync_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Csync::new");
    }
    size_t channels() const { return c_; }
    // phase (2^-64 turn) and frequency (2^-40 turn per symbol) of one channel's next symbol
    std::pair<uint64_t, int64_t> state(size_t k) {
        uint64_t ph = 0;
        int64_t f = 0;
        check(sdr_csync_get_state(h_, k, &ph, &f), "Csync::state");
        return {ph, f};
    }
    // in: channels rows, row k of n_in[k] symbols at row stride in_stride (>= the longest row)
    Out process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride) {
        const size_t cap = std::max<size_t>(1, *std::max_element(n_in.begin(), n_in.end()));
        std::vector<Complex> sym(cap * c_);
        std::vector<uint64_t> ph(cap * c_);
        std::vector<float> err(cap * c_);
        check(sdr_csync_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                                reinterpret_cast<float *>(sym.data()), ph.data(), err.data(), cap),
              "Csync::process");
        Out o;
        o.sym.resize(c_);
        o.phase.resize(c_);
        o.err.resize(c_);
        for (size_t k = 0; k < c_; ++k) {
            o.sym[k].assign(sym.begin() + k * cap, sym.begin() + k * cap + n_in[k]);
            o.phase[k].assign(ph.begin() + k * cap, ph.begin() + k * cap + n_in[k]);
            o.err[k].assign(err.begin() + k * cap, err.begin() + k * cap + n_in[k]);
        }
        return o;
    }
    void reset() { check(sdr_csync_reset(h_), "Csync::reset"); }
};

// Adaptive equalizer bank (sdr_eq): an N-tap FIR per channel whose complex weights adapt by blind CMA and then
// decision-directed LMS.  Channel k: an adaptation set {order, mu, radius, err_max, cma_symbols} (symbols s <
// cma_symbols adapt by CMA, later ones by DD) and initial taps (none: the centre spike); each call returns one
// equalized symbol per input symbol with its error.
class Eq : public Handle<sdr_eq_t, sdr_eq_destroy, sdr_eq_clone> {
    size_t c_ = 0, n_ = 0;

  public:
    struct Out {
        std::vector<std::vector<Complex>> sym;
        std::vector<std::vector<Complex>> err;
    };
    // adapt: one (shared) or one per channel; taps: empty (centre spike), n_taps (shared) or channels * n_taps
    Eq(size_t n_taps, size_t channels, const std::vector<sdr_eq_adapt_t> &adapt, const std::vector<Complex> &taps = {})
        : c_(channels), n_(n_taps) {
        if (n_taps == 0 || taps.size() % n_taps != 0) throw sdr::Error(SDR_ERR_INVALID_ARG, "Eq::new");
        sdr_eq_config_t cfg{};
        cfg.n_taps = n_;
        cfg.taps = taps.empty() ? nullptr : reinterpret_cast<const float *>(taps.data());
        cfg.n_tap_sets = taps.size() / n_taps;
        cfg.adapt = adapt.data();
        cfg.n_adapt = adapt.size();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_eq_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Eq::new");
    }
    size_t channels() const { return c_; }
    size_t taps_per_channel() const { return n_; }
    // the taps of one channel for its next symbol
    std::vector<Complex> taps(size_t k) {
        std::vector<Complex> w(n_);
        check(sdr_eq_get_taps(h_, k, reinterpret_cast<float *>(w.data())), "Eq::taps");
        return w;
    }
    // in: channels rows, row k of n_in[k] symbols at row stride in_stride (>= the longest row)
    Out process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride) {
        const size_t cap = std::max<size_t>(1, *std::max_element(n_in.begin(), n_in.end()));
        std::vector<Complex> sym(cap * c_), err(cap * c_);
        check(sdr_eq_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                             reinterpret_cast<float *>(sym.data()), reinterpret_cast<float *>(err.data()), cap),
              "Eq::process");
        Out o;
        o.sym.resize(c_);
        o.err.resize(c_);
        for (size_t k = 0; k < c_; ++k) {
            o.sym[k].assign(sym.begin() + k * cap, sym.begin() + k * cap + n_in[k]);
            o.err[k].assign(err.begin() + k * cap, err.begin() + k * cap + n_in[k]);
        }
        return o;
    }
    void reset() { check(sdr_eq_reset(h_), "Eq::reset"); }
};

struct BiquadD {  // biquad.rs:74-81 + simple.rs Identity
    sdr_biquad_design_t d;
    static BiquadD LowPass(float f, float q) { return {{SDR_BQ_LOWPASS, f, q}}; }
    static BiquadD HighPass(float f, float q) { return {{SDR_BQ_HIGHPASS, f, q}}; }
    static BiquadD BandPass(float f, float q) { return {{SDR_BQ_BANDPASS, f, q}}; }
    static BiquadD Notch(float f, float q) { return {{SDR_BQ_NOTCH, f, q}}; }
    static BiquadD Lr(float decayrate) { return {{SDR_BQ_LR, decayrate, 0.0f}}; }
    static BiquadD Identity() { return {{SDR_BQ_IDENTITY, 0.0f, 0.0f}}; }
};

// Biquad<f32, A> (biquad.rs:5-71) as a block stream filter; BiquadD::design(rate) (biquad.rs:83-154) builds it
template <class A>
class Biquad : public Handle<sdr_biquad_t, sdr_biquad_destroy, sdr_biquad_clone> {

  public:
    Biquad(const BiquadD &d, float rate) {
        sdr_biquad_config_t cfg{};
        cfg.designs = &d.d;
        cfg.n_designs = 1;
        cfg.n_streams = 1;
        cfg.rate = rate;
        cfg.sample_complex = SampleTraits<A>::channels == 2;
        int err = 0;
        h_ = sdr_biquad_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "BiquadD::design");
    }
    void process(const A *in, size_t n, std::vector<A> &out) {
        out.resize(n);
        check(sdr_biquad_process(h_, reinterpret_cast<const float *>(in), n, n, reinterpret_cast<float *>(out.data()), n),
              "Biquad::apply");
    }
    void reset() { check(sdr_biquad_reset(h_), "Biquad::reset"); }
};

class Pll;
struct PllDesign {  // pll.rs:4-36
    float reference, gain;
    BiquadD loopfilter, outputfilter, lockfilter;
    PllDesign(float reference_, float gain_, BiquadD loop, BiquadD output, BiquadD lock)
        : reference(reference_), gain(gain_), loopfilter(loop), outputfilter(output), lockfilter(lock) {}
    Pll design(float rate) const;  // FilterDesign::design (pll.rs:48-60)
};

class Pll : public Handle<sdr_pll_t, sdr_pll_destroy, sdr_pll_clone> {  // pll.rs:13-85 ; Output = Option<f32>

  public:
    Pll(const PllDesign &d, float rate, unsigned flags = 0) {
        sdr_pll_design_t cd{d.reference, d.gain, d.loopfilter.d, d.outputfilter.d, d.lockfilter.d};
        sdr_pll_config_t cfg{};
        cfg.designs = &cd;
        cfg.n_designs = 1;
        cfg.n_streams = 1;
        cfg.rate = rate;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_pll_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "PllDesign::design");
    }
    void process(const Complex *in, size_t n, std::vector<std::optional<float>> &out) {
        std::vector<float> v(n);
        std::vector<uint8_t> lk(n);
        check(sdr_pll_process(h_, reinterpret_cast<const float *>(in), n, n, v.data(), lk.data(), n), "Pll::process");
        out.resize(n);
        for (size_t i = 0; i < n; ++i) out[i] = lk[i] ? std::optional<float>(v[i]) : std::nullopt;
    }
    std::optional<float> apply(Complex value) {
        std::vector<std::optional<float>> o;
        process(&value, 1, o);
        return o[0];
    }
    // the closure of main.rs:62-71 with this Pll as `pllpilot`: v -> (mono, diff)
    void stereo_decode(const float *v, size_t n, std::vector<std::pair<float, float>> &out) {
        out.resize(n);
        check(sdr_pll_stereo_decode(h_, v, n, n, reinterpret_cast<float *>(out.data()), n), "Pll::stereo_decode");
    }
    float nphase() { float a, b, c; check(sdr_pll_get_state(h_, 0, &a, &b, &c), "Pll::nphase"); return a; }  // pub nphase
    Complex value() { float a, b, c; check(sdr_pll_get_state(h_, 0, &a, &b, &c), "Pll::value"); return {b, c}; }  // pub value
};
inline Pll PllDesign::design(float rate) const { return Pll(*this, rate); }

}  // namespace filter

// =========================================================================================
namespace signal {

inline size_t decimate_wait(float rate_in, float rate_out) { return sdr_decimate_wait(rate_in, rate_out); }

// A Signal yields blocks: next_block appends up to n samples to `out` and returns how many (0 = end).
template <class SampleT>
class Signal : public std::enable_shared_from_this<Signal<SampleT>> {
  public:
    using Sample = SampleT;
    virtual ~Signal() = default;
    virtual size_t next_block(size_t n, std::vector<Sample> &out) = 0;
    virtual float rate() const = 0;
    // rtl_tcp sources can hand out raw bytes so the consumer kernel unpacks on the GPU
    virtual bool has_raw_u8iq() const { return false; }
    virtual size_t next_raw(size_t, std::vector<uint8_t> &) { return 0; }

    std::vector<Sample> collect(size_t block = (size_t)1 << 20) {  // .iter().collect()
        std::vector<Sample> all, b;
        for (;;) {
            b.clear();
            if (next_block(block, b) == 0) break;
            all.insert(all.end(), b.begin(), b.end());
        }
        return all;
    }
};
template <class A> using Sig = std::shared_ptr<Signal<A>>;

template <class A>
class FromIter : public Signal<A> {  // sources.rs:6-36
    std::vector<A> data_;
    size_t pos_ = 0;
    float rate_;

  public:
    FromIter(float rate, std::vector<A> d) : data_(std::move(d)), rate_(rate) {}
    size_t next_block(size_t n, std::vector<A> &out) override {
        const size_t k = std::min(n, data_.size() - pos_);
        out.insert(out.end(), data_.begin() + pos_, data_.begin() + pos_ + k);
        pos_ += k;
        return k;
    }
    float rate() const override { return rate_; }
};
template <class A> Sig<A> from_iter(float rate, std::vector<A> d) { return std::make_shared<FromIter<A>>(rate, std::move(d)); }

class RtlTcpBytes : public Signal<Complex> {  // RtlTcpSignal (rtltcp.rs:151-168) over a captured byte buffer
    std::vector<uint8_t> raw_;
    size_t pos_ = 0;  // samples
    float rate_;

  public:
    RtlTcpBytes(float rate, std::vector<uint8_t> raw) : raw_(std::move(raw)), rate_(rate) {}
    bool has_raw_u8iq() const override { return true; }
    size_t next_raw(size_t n, std::vector<uint8_t> &out) override {
        const size_t k = std::min(n, raw_.size() / 2 - pos_);
        out.insert(out.end(), raw_.begin() + 2 * pos_, raw_.begin() + 2 * (pos_ + k));
        pos_ += k;
        return k;
    }
    size_t next_block(size_t n, std::vector<Complex> &out) override {
        std::vector<uint8_t> b;
        const size_t k = next_raw(n, b);
        if (!k) return 0;
        const size_t o = out.size();
        out.resize(o + k);
        check(sdr_unpack_u8iq(b.data(), k, reinterpret_cast<float *>(out.data() + o), 0), "RtlTcpSignal::next");
        return k;
    }
    float rate() const override { return rate_; }
};
inline Sig<Complex> from_u8iq(float rate, std::vector<uint8_t> raw) { return std::make_shared<RtlTcpBytes>(rate, std::move(raw)); }

// signal::Filter (adapters/mod.rs:67-100) for a Fir design; decimation > 1 = Filter followed by Decimate, fused
template <class C, class A>
class FirFilter : public Signal<A> {
    Sig<A> up_;
    std::vector<C> taps_;
    size_t D_;
    std::unique_ptr<filter::Fir<C, A>> fir_;
    bool raw_;

  public:
    FirFilter(Sig<A> up, std::vector<C> taps, size_t D = 1) : up_(std::move(up)), taps_(std::move(taps)), D_(D) {
        raw_ = std::is_same<A, Complex>::value && up_->has_raw_u8iq();
    }
    const std::vector<C> &taps() const { return taps_; }
    Sig<A> upstream() const { return up_; }
    bool started() const { return (bool)fir_; }
    size_t next_block(size_t n, std::vector<A> &out) override {
        if (!fir_) fir_.reset(new filter::Fir<C, A>(taps_, D_, raw_));
        for (;;) {
            std::vector<A> y;
            if (raw_) {
                std::vector<uint8_t> b;
                const size_t k = up_->next_raw(n * D_, b);
                if (!k) return 0;
                fir_->process(b.data(), k, y);
            } else {
                std::vector<A> x;
                const size_t k = up_->next_block(n * D_, x);
                if (!k) return 0;
                fir_->process(x.data(), k, y);
            }
            if (y.empty()) continue;
            out.insert(out.end(), y.begin(), y.end());
            return y.size();
        }
    }
    float rate() const override { return up_->rate(); }
};

// signal::Decimate (adapters/mod.rs:14-41); rate() is the upstream rate (:38-40, reference quirk)
template <class A>
class Decimate : public Signal<A> {
    Sig<A> up_;
    size_t wait_, phase_ = 0;

  public:
    Decimate(Sig<A> up, float rate) : up_(std::move(up)) {
        wait_ = decimate_wait(up_->rate(), rate);
        if (wait_ == 0) throw sdr::Error(SDR_ERR_INVALID_ARG, "Decimate (wait == 0 underflows in the reference)");
    }
    size_t wait() const { return wait_; }
    size_t next_block(size_t n, std::vector<A> &out) override {
        for (;;) {
            std::vector<A> x;
            const size_t k = up_->next_block(n * wait_, x);
            if (!k) return 0;
            size_t made = 0;
            for (size_t i = wait_ - 1 - phase_; i < k; i += wait_) { out.push_back(x[i]); ++made; }
            phase_ = (phase_ + k) % wait_;
            if (made) return made;
        }
    }
    float rate() const override { return up_->rate(); }
};

// signal::Resample (adapters/resample.rs:5-86)
template <class A>
class Resample : public Signal<A> {
    Sig<A> up_;
    resample::SampleRate<A> sr_;
    float rate_;
    double ratio_;
    std::vector<A> buffer_, resampled_;
    size_t buffer_size_ = 4096, next_ = 4096;
    bool done_ = false;

  public:
    Resample(Sig<A> up, resample::ConverterType typ, float rate)
        : up_(std::move(up)), sr_(typ), rate_(rate), ratio_((double)rate / (double)up_->rate()) {
        buffer_.reserve(buffer_size_);
        resampled_.reserve(buffer_size_);
    }
    size_t next_block(size_t n, std::vector<A> &out) override {
        size_t made = 0;
        while (made < n) {
            if (done_) break;
            while (next_ >= resampled_.size()) {
                if (buffer_.size() < buffer_size_) up_->next_block(buffer_size_ - buffer_.size(), buffer_);  // refill (:46-52)
                resampled_.reserve(buffer_size_);
                const size_t used = sr_.process(ratio_, buffer_, resampled_);                              // (:55-59)
                if (buffer_.empty() && resampled_.empty()) { done_ = true; break; }                          // (:62-65)
                buffer_.erase(buffer_.begin(), buffer_.begin() + used);                                      // (:68)
                if (resampled_.empty()) continue;                                                            // (:70-73)
                next_ = 0;
            }
            if (done_) break;
            const size_t k = std::min(n - made, resampled_.size() - next_);
            out.insert(out.end(), resampled_.begin() + next_, resampled_.begin() + next_ + k);
            next_ += k;
            made += k;
            if (made) break;  // hand back what one chunk produced; callers loop
        }
        return made;
    }
    float rate() const override { return rate_; }
};

template <class A>
class Take : public Signal<A> {  // adapters/mod.rs:241-268
    Sig<A> up_;
    size_t left_;

  public:
    Take(Sig<A> up, float duration) : up_(std::move(up)) { left_ = sdr_duration_samples(up_->rate(), duration); }
    size_t next_block(size_t n, std::vector<A> &out) override {
        n = std::min(n, left_);
        if (!n) return 0;
        const size_t k = up_->next_block(n, out);
        left_ -= k;
        return k;
    }
    float rate() const override { return up_->rate(); }
};

template <class A>
class Skip : public Signal<A> {  // adapters/mod.rs:166-194
    Sig<A> up_;
    size_t left_;

  public:
    Skip(Sig<A> up, float duration) : up_(std::move(up)) { left_ = sdr_duration_samples(up_->rate(), duration); }
    size_t next_block(size_t n, std::vector<A> &out) override {
        while (left_ > 0) {
            std::vector<A> junk;
            const size_t k = up_->next_block(std::min<size_t>(left_, 1 << 20), junk);
            if (!k) return 0;
            left_ -= k;
        }
        return up_->next_block(n, out);
    }
    float rate() const override { return up_->rate(); }
};

// signal::Block (adapters/block.rs:106-207).  The upstream is pulled in blocks of ceil(size * rate) samples (:117),
// one block ahead of the reader (target = 1, :165-189); clone() is a tee (:129-140): clones share the upstream and one
// deque of blocks with a per-reader `available` count (TeeDeque, :7-103) -- a new reader starts with available =
// data.len(), so it also sees the blocks the deque still held.  Faithful to the reference's quirk that `next` returns
// current[0] without advancing `i` when it moves to a new block (:197-199): the first sample of every block is
// delivered twice unless dedup is set (a deliberate divergence).
template <class A>
class Block : public Signal<A> {
    struct Shared {
        Sig<A> up;
        std::deque<std::vector<A>> data;   // samples; newest block at the front
        std::deque<std::vector<uint8_t>> raw;  // same blocks as raw rtl_tcp bytes when the upstream hands those out
        std::vector<size_t> available{0};
        size_t block_size = 0;
        bool is_raw = false, dedup = false;
        float rate = 0.0f;
    };
    std::shared_ptr<Shared> sh_;
    size_t id_ = 0, i_ = 0, cur_len_ = 0;
    std::vector<A> cur_;
    std::vector<uint8_t> cur_raw_;
    bool have_cur_ = false;

    void push() {  // TeeDequePush::push (:76-89) around the fill closure (:176-187)
        Shared &s = *sh_;
        const size_t held = s.is_raw ? s.raw.size() : s.data.size();
        if (*std::max_element(s.available.begin(), s.available.end()) < held) {
            if (s.is_raw) s.raw.pop_back(); else s.data.pop_back();
        }
        if (s.is_raw) { std::vector<uint8_t> v; s.up->next_raw(s.block_size, v); s.raw.push_front(std::move(v)); }
        else { std::vector<A> v; s.up->next_block(s.block_size, v); s.data.push_front(std::move(v)); }
        for (auto &a : s.available) ++a;
    }
    void load(size_t idx) {
        Shared &s = *sh_;
        if (s.is_raw) { cur_raw_ = s.raw[idx]; cur_len_ = cur_raw_.size() / 2; }
        else { cur_ = s.data[idx]; cur_len_ = cur_.size(); }
    }
    size_t fetch() {  // the else-branch of Block::next (:154-195)
        Shared &s = *sh_;
        cur_.clear(); cur_raw_.clear(); cur_len_ = 0; i_ = 0;
        bool needs_extra = true;
        size_t avail = 0;
        if (s.available[id_] > 0) { avail = --s.available[id_]; load(avail); needs_extra = false; }
        if (avail < 1) {
            const size_t jobs = 1 - avail + (needs_extra ? 1 : 0);
            for (size_t j = 0; j < jobs; ++j) push();
            if (needs_extra) load(--s.available[id_]);
        }
        have_cur_ = true;
        return cur_len_;
    }
    template <class V, class T>
    size_t serve(size_t n, std::vector<T> &out, const V &cur, size_t per) {
        size_t made = 0;
        if (!have_cur_ || i_ >= cur_len_) {
            // note: fetch() re-fills `cur`, which the caller passed by reference
            if (fetch() == 0 || n == 0) return 0;
            if (!sh_->dedup) { out.insert(out.end(), cur.begin(), cur.begin() + per); made = 1; }  // (:197-199)
        }
        const size_t k = std::min(n - made, cur_len_ - i_);
        out.insert(out.end(), cur.begin() + per * i_, cur.begin() + per * (i_ + k));
        i_ += k;
        return made + k;
    }

  public:
    Block(Sig<A> up, float size, bool dedup = false) : sh_(std::make_shared<Shared>()) {
        sh_->rate = up->rate();
        sh_->block_size = sdr_block_samples(size, up->rate());
        sh_->is_raw = up->has_raw_u8iq();
        sh_->dedup = dedup;
        sh_->up = std::move(up);
    }
    // Clone for Block (:129-140) + Clone for TeeDeque (:92-103)
    std::shared_ptr<Block<A>> clone() const {
        auto b = std::shared_ptr<Block<A>>(new Block<A>(*this));
        b->cur_.clear(); b->cur_raw_.clear(); b->cur_len_ = 0; b->i_ = 0; b->have_cur_ = false;
        Shared &s = *sh_;
        s.available.push_back(s.is_raw ? s.raw.size() : s.data.size());
        b->id_ = s.available.size() - 1;
        return b;
    }
    size_t block_size() const { return sh_->block_size; }
    size_t next_block(size_t n, std::vector<A> &out) override {
        if (!sh_->is_raw) return serve(n, out, cur_, 1);
        // raw upstream, sample consumer: unpack the served bytes (RtlTcpSignal::next, rtltcp.rs:158-164)
        std::vector<uint8_t> b;
        const size_t k = serve(n, b, cur_raw_, 2);
        if (!k) return 0;
        const size_t o = out.size();
        out.resize(o + k);
        if (std::is_same<A, Complex>::value)
            check(sdr_unpack_u8iq(b.data(), k, reinterpret_cast<float *>(out.data() + o), 0), "Block::next");
        return k;
    }
    bool has_raw_u8iq() const override { return sh_->is_raw; }
    size_t next_raw(size_t n, std::vector<uint8_t> &out) override { return serve(n, out, cur_raw_, 2); }
    float rate() const override { return sh_->rate; }
};

template <class A, class B>
class Map : public Signal<B> {  // adapters/mod.rs:139-163
    Sig<A> up_;
    std::function<B(A)> f_;

  public:
    Map(Sig<A> up, std::function<B(A)> f) : up_(std::move(up)), f_(std::move(f)) {}
    size_t next_block(size_t n, std::vector<B> &out) override {
        std::vector<A> x;
        const size_t k = up_->next_block(n, x);
        for (size_t i = 0; i < k; ++i) out.push_back(f_(x[i]));
        return k;
    }
    float rate() const override { return up_->rate(); }
};

// ---- the combinators of trait Signal (src/signal/mod.rs:18-122) as free functions over Sig<A> ----
template <class A, class C> Sig<A> filter(Sig<A> s, std::vector<C> taps) { return std::make_shared<FirFilter<C, A>>(std::move(s), std::move(taps)); }
template <class A> Sig<A> decimate(Sig<A> s, float rate) {
    // Filter followed by Decimate: fuse so only kept outputs are computed
    if (auto f = std::dynamic_pointer_cast<FirFilter<float, A>>(s))
        if (!f->started()) return std::make_shared<FirFilter<float, A>>(f->upstream(), f->taps(), decimate_wait(s->rate(), rate));
    if (auto f = std::dynamic_pointer_cast<FirFilter<Complex, A>>(s))
        if (!f->started()) return std::make_shared<FirFilter<Complex, A>>(f->upstream(), f->taps(), decimate_wait(s->rate(), rate));
    return std::make_shared<Decimate<A>>(std::move(s), rate);
}
template <class A> Sig<A> resample_with(Sig<A> s, resample::ConverterType typ, float rate) { return std::make_shared<Resample<A>>(std::move(s), typ, rate); }
template <class A> Sig<A> resample(Sig<A> s, float rate) { return resample_with(std::move(s), resample::ConverterType::SincBestQuality, rate); }  // mod.rs:83
template <class A> Sig<A> take(Sig<A> s, float duration) { return std::make_shared<Take<A>>(std::move(s), duration); }
template <class A> Sig<A> skip(Sig<A> s, float duration) { return std::make_shared<Skip<A>>(std::move(s), duration); }
template <class A> std::shared_ptr<Block<A>> block(Sig<A> s, float size, bool dedup = false) { return std::make_shared<Block<A>>(std::move(s), size, dedup); }
template <class A, class F> auto map(Sig<A> s, F f) -> Sig<decltype(f(std::declval<A>()))> {
    using B = decltype(f(std::declval<A>()));
    return std::make_shared<Map<A, B>>(std::move(s), std::function<B(A)>(f));
}

}  // namespace signal

// =========================================================================================
namespace fft {

// fft::fft (src/fft.rs:3-28): drains the signal, one N-point transform, (label, value) pairs
inline std::vector<std::pair<float, Complex>> fft(signal::Sig<Complex> input) {
    const float rate = input->rate();
    std::vector<std::pair<float, Complex>> collated;
    sdr_fft_config_t cfg{};
    cfg.flags = SDR_FFT_SHIFT | SDR_FFT_NORM;
    std::vector<uint8_t> raw;
    std::vector<Complex> data;
    const void *src;
    if (input->has_raw_u8iq()) {
        input->next_raw((size_t)1 << 62, raw);
        cfg.n = raw.size() / 2;
        cfg.input_format = SDR_FMT_U8IQ;
        src = raw.data();
    } else {
        data = input->collect();
        cfg.n = data.size();
        cfg.input_format = SDR_FMT_C64;
        src = data.data();
    }
    if (cfg.n == 0) return collated;
    int err = 0;
    sdr_fft_t *plan = sdr_fft_create(&cfg, &err);
    if (!plan) throw Error(err, "fft::fft");
    std::vector<Complex> vals(cfg.n);
    std::vector<float> labels(cfg.n);
    const int rc = sdr_fft_exec(plan, src, 1, reinterpret_cast<float *>(vals.data()));
    sdr_fft_destroy(plan);
    check(rc, "fft::fft");
    check(sdr_fft_labels(cfg.n, rate, 0, labels.data()), "fft::fft labels");
    collated.reserve(cfg.n);
    for (size_t i = 0; i < cfg.n; ++i) collated.emplace_back(labels[i], vals[i]);
    return collated;
}

// fft::rfft (src/fft.rs:30-37)
inline std::vector<std::pair<float, Complex>> rfft(signal::Sig<float> input) {
    const float rate = input->rate();
    std::vector<float> data = input->collect();
    std::vector<std::pair<float, Complex>> collated;
    if (data.empty()) return collated;
    sdr_fft_config_t cfg{};
    cfg.n = data.size();
    cfg.input_format = SDR_FMT_F32;
    cfg.flags = SDR_FFT_SHIFT | SDR_FFT_NORM | SDR_FFT_RFFT;
    int err = 0;
    sdr_fft_t *plan = sdr_fft_create(&cfg, &err);
    if (!plan) throw Error(err, "fft::rfft");
    const size_t keep = sdr_fft_output_len(plan);
    std::vector<Complex> vals(keep);
    std::vector<float> labels(keep);
    const int rc = sdr_fft_exec(plan, data.data(), 1, reinterpret_cast<float *>(vals.data()));
    sdr_fft_destroy(plan);
    check(rc, "fft::rfft");
    check(sdr_fft_labels(cfg.n, rate, 1, labels.data()), "fft::rfft labels");
    for (size_t i = 0; i < keep; ++i) collated.emplace_back(labels[i], vals[i]);
    return collated;
}

// signal.window(duration).decimate(fps).map(|w| fft::fft(w)) of examples/live.rs:30-39 behind sdr_window_fft_*:
// feed blocks of samples, get the kept windows' spectra (each `window()` values, shifted and 1/sqrt(N)-scaled like
// fft::fft) back to back.  window = (duration * rate).round() (adapters/mod.rs:279), hop = Decimate's wait (mod.rs:22).
class WindowSpectra {
    sdr_window_fft_t *h_ = nullptr;
    size_t n_ = 0;

  public:
    WindowSpectra(float rate, float duration, float fps, bool u8iq = false) {
        sdr_window_fft_config_t cfg{};
        cfg.window = sdr_duration_samples(rate, duration);
        cfg.hop = sdr_decimate_wait(rate, fps);
        cfg.input_format = u8iq ? SDR_FMT_U8IQ : SDR_FMT_C64;
        cfg.flags = SDR_FFT_SHIFT | SDR_FFT_NORM;
        int err = 0;
        h_ = sdr_window_fft_create(&cfg, &err);
        if (!h_) throw Error(err, "WindowSpectra::new");
        n_ = cfg.window;
    }
    WindowSpectra(const WindowSpectra &) = delete;
    WindowSpectra &operator=(const WindowSpectra &) = delete;
    ~WindowSpectra() { sdr_window_fft_destroy(h_); }
    size_t window() const { return n_; }
    // in: n samples (Complex, or 2n bytes when constructed with u8iq); returns the number of spectra appended to out
    size_t process(const void *in, size_t n, std::vector<Complex> &out) {
        const size_t nw = sdr_window_fft_output_count(h_, n);
        const size_t at = out.size();
        out.resize(at + nw * n_);
        size_t got = 0;
        Complex dummy;
        check(sdr_window_fft_process(h_, in, n, reinterpret_cast<float *>(nw ? out.data() + at : &dummy), nw, &got),
              "WindowSpectra::process");
        return got;
    }
};

// window -> decimate -> map(fft::fft) -> |.|^2 -> mean of `average` behind sdr_psd_*: feed blocks of samples, get the
// averaged power spectra (n floats each, bins shifted like fft::fft, scaled 1/n like its 1/sqrt(n)) back to back.
// taper: n real values or empty (rectangular).  Copies with sdr_psd_clone.
class PowerSpectra : public Handle<sdr_psd_t, sdr_psd_destroy, sdr_psd_clone> {
    size_t n_ = 0;

  public:
    PowerSpectra(size_t n, size_t hop, size_t average, const std::vector<float> &taper = {}, bool u8iq = false,
                 unsigned flags = SDR_PSD_SHIFT | SDR_PSD_NORM)
        : n_(n) {
        if (!taper.empty() && taper.size() != n) throw Error(SDR_ERR_INVALID_ARG, "PowerSpectra::new");
        sdr_psd_config_t cfg{};
        cfg.n = n;
        cfg.hop = hop;
        cfg.average = average;
        cfg.window = taper.empty() ? nullptr : taper.data();
        cfg.input_format = u8iq ? SDR_FMT_U8IQ : SDR_FMT_C64;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_psd_create(&cfg, &err);
        if (!h_) throw Error(err, "PowerSpectra::new");
    }
    size_t bins() const { return n_; }
    int last_path() const { return sdr_psd_last_path(h_); }
    // in: n samples (Complex, or 2n bytes when constructed with u8iq); returns the number of spectra appended to out
    size_t process(const void *in, size_t n, std::vector<float> &out) {
        const size_t ns = sdr_psd_output_count(h_, n);
        const size_t at = out.size();
        out.resize(at + ns * n_);
        size_t got = 0;
        float dummy;
        check(sdr_psd_process(h_, in, n, ns ? out.data() + at : &dummy, ns, n_, &got), "PowerSpectra::process");
        return got;
    }
    void reset() { check(sdr_psd_reset(h_), "PowerSpectra::reset"); }
};

}  // namespace fft

// =========================================================================================
namespace fec {

// Viterbi decoder bank (sdr_vit): soft-decision decoding of C streams of one rate-1/n convolutional code (constraint
// length K, generators in the octal convention, decision depth L).  Each call takes n floats per step (positive
// favours bit 0) and returns the bits it releases, one byte (0 or 1) each; finish releases the rest.
class Vit : public Handle<sdr_vit_t, sdr_vit_destroy, sdr_vit_clone> {
    size_t c_ = 0, n_ = 0, l_ = 0;

    static std::vector<std::vector<uint8_t>> rows(const std::vector<uint8_t> &buf, size_t stride,
                                                  const std::vector<size_t> &got) {
        std::vector<std::vector<uint8_t>> o(got.size());
        for (size_t k = 0; k < got.size(); ++k) o[k].assign(buf.begin() + k * stride, buf.begin() + k * stride + got[k]);
        return o;
    }

  public:
    // scale: one (shared) or one per channel
    Vit(unsigned K, const std::vector<uint32_t> &gens, size_t depth, const std::vector<float> &scale, size_t channels,
        bool zero_start = true)
        : c_(channels), n_(gens.size()), l_(depth) {
        sdr_vit_config_t cfg{};
        cfg.constraint = K;
        cfg.gens = gens.data();
        cfg.n_gens = gens.size();
        cfg.depth = depth;
        cfg.scale = scale.data();
        cfg.n_scales = scale.size();
        cfg.zero_start = zero_start ? 1 : 0;
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_vit_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Vit::new");
    }
    size_t channels() const { return c_; }
    // the bits a call of n_in steps per channel releases
    std::vector<size_t> output_count(const std::vector<size_t> &n_in) const {
        std::vector<size_t> o(c_);
        check(sdr_vit_output_count(h_, n_in.data(), o.data()), "Vit::output_count");
        return o;
    }
    // in: channels rows, row k of n_in[k] steps of n floats at a row stride of in_stride steps (>= the longest row)
    std::vector<std::vector<uint8_t>> process(const float *in, const std::vector<size_t> &n_in, size_t in_stride) {
        const std::vector<size_t> cnt = output_count(n_in);
        const size_t cap = (std::max<size_t>(4, *std::max_element(cnt.begin(), cnt.end())) + 3) & ~(size_t)3;
        std::vector<uint8_t> buf(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_vit_process(h_, in, n_in.data(), in_stride, buf.data(), cap, got.data()), "Vit::process");
        return rows(buf, cap, got);
    }
    // the remaining bits of every channel (traced back from state 0 when terminated); the bank returns to its start
    std::vector<std::vector<uint8_t>> finish(bool terminated) {
        const size_t cap = l_ + 32;
        std::vector<uint8_t> buf(cap * c_);
        std::vector<size_t> got(c_);
        check(sdr_vit_finish(h_, nullptr, terminated ? 1 : 0, buf.data(), cap, got.data()), "Vit::finish");
        return rows(buf, cap, got);
    }
    void reset() { check(sdr_vit_reset(h_), "Vit::reset"); }
};

// frame synchronizer bank: per channel, finds the sync word, locks to the frames and emits their payloads derotated
class Fsync : public Handle<sdr_fsync_t, sdr_fsync_destroy, sdr_fsync_clone> {
    size_t c_ = 0;

  public:
    struct Out {
        std::vector<std::vector<Complex>> payload;
        std::vector<std::vector<sdr_fsync_record_t>> records;
    };
    // words: one row of Lp symbols (shared) or one per channel; params: one (shared) or one per channel
    Fsync(size_t channels, size_t word_len, const std::vector<Complex> &words,
          const std::vector<sdr_fsync_params_t> &params)
        : c_(channels) {
        sdr_fsync_config_t cfg{};
        cfg.word_len = word_len;
        cfg.words = reinterpret_cast<const float *>(words.data());
        cfg.n_words = word_len ? words.size() / word_len : 0;
        cfg.params = params.data();
        cfg.n_params = params.size();
        cfg.n_channels = c_;
        int err = 0;
        h_ = sdr_fsync_create(&cfg, &err);
        if (!h_) throw sdr::Error(err, "Fsync::new");
    }
    size_t channels() const { return c_; }
    // (payload, record) bounds per channel for the next n_in[k] symbols
    std::pair<std::vector<size_t>, std::vector<size_t>> max_output(const std::vector<size_t> &n_in) const {
        std::vector<size_t> p(c_), r(c_);
        check(sdr_fsync_max_output(h_, n_in.data(), p.data(), r.data()), "Fsync::max_output");
        return {p, r};
    }
    sdr_fsync_state_t state(size_t k) {
        sdr_fsync_state_t s{};
        check(sdr_fsync_get_state(h_, k, &s), "Fsync::state");
        return s;
    }
    // in: channels rows, row k of n_in[k] symbols at row stride in_stride (>= the longest row)
    Out process(const Complex *in, const std::vector<size_t> &n_in, size_t in_stride) {
        const auto caps = max_output(n_in);
        const size_t cap = std::max<size_t>(1, *std::max_element(caps.first.begin(), caps.first.end()));
        const size_t rcap = std::max<size_t>(1, *std::max_element(caps.second.begin(), caps.second.end()));
        std::vector<Complex> pay(cap * c_);
        std::vector<sdr_fsync_record_t> rec(rcap * c_);
        std::vector<size_t> got(c_), rgot(c_);
        check(sdr_fsync_process(h_, reinterpret_cast<const float *>(in), n_in.data(), in_stride,
                                reinterpret_cast<float *>(pay.data()), cap, cap, got.data(), rec.data(), rcap, rcap,
                                rgot.data()),
              "Fsync::process");
        Out o;
        o.payload.resize(c_);
        o.records.resize(c_);
        for (size_t k = 0; k < c_; ++k) {
            o.payload[k].assign(pay.begin() + k * cap, pay.begin() + k * cap + got[k]);
            o.records[k].assign(rec.begin() + k * rcap, rec.begin() + k * rcap + rgot[k]);
        }
        return o;
    }
    void reset() { check(sdr_fsync_reset(h_), "Fsync::reset"); }
};

}  // namespace fec

// =========================================================================================
namespace app {

// The receiver of src/main.rs:32-81 as one device-resident pipeline (sdr_fm_*): rtl_tcp bytes in, 48 kHz
// (left, right) frames out; a batch of stations shares every launch.
class FmStereo {
    sdr_fm_t *h_ = nullptr;
    size_t n_st_;

  public:
    explicit FmStereo(size_t n_stations = 1, float rate = 1800000.0f, unsigned flags = 0) : n_st_(n_stations) {
        sdr_fm_config_t cfg{};
        cfg.n_stations = n_stations;
        cfg.rate = rate;
        cfg.flags = flags;
        int err = 0;
        h_ = sdr_fm_create(&cfg, &err);
        if (!h_) throw Error(err, "FmStereo::new");
    }
    FmStereo(const FmStereo &) = delete;
    FmStereo &operator=(const FmStereo &) = delete;
    ~FmStereo() { sdr_fm_destroy(h_); }
    float rate() const { return sdr_fm_output_rate(h_); }
    // iq: n_stations rows of 2n bytes; out: n_stations rows of the returned number of frames
    size_t process(const uint8_t *iq, size_t n, bool end_of_input, std::vector<std::pair<float, float>> &out) {
        const size_t cap = sdr_fm_max_output(h_, n);
        out.resize(n_st_ * cap);
        size_t got = 0;
        check(sdr_fm_process(h_, iq, n, 2 * n, reinterpret_cast<float *>(out.data()), cap, cap, &got, end_of_input ? 1 : 0),
              "FmStereo::process");
        if (got != cap)
            for (size_t s = 1; s < n_st_; ++s) std::copy(out.begin() + s * cap, out.begin() + s * cap + got, out.begin() + s * got);
        out.resize(n_st_ * got);
        return got;
    }
    void reset() { check(sdr_fm_reset(h_), "FmStereo::reset"); }
};

}  // namespace app
}  // namespace sdr

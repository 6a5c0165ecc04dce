"""Operator handles over the C ABI.  Names follow the reference crate:

    filter::Fir          (src/filter/fir.rs)           -> Fir
    filter::PllDesign    (src/filter/pll.rs)           -> PllDesign / PllBatch
    filter::BiquadD      (src/filter/biquad.rs)        -> BiquadD
    resample::SampleRate (src/resample.rs)             -> SampleRate, ConverterType
    fft::fft / rfft      (src/fft.rs)                  -> FftPlan, fft(), rfft()

Host entry points take numpy arrays; `*_dev` entry points take anything with .data_ptr()
(torch CUDA tensors) or raw integer device addresses and run asynchronously on the handle's stream.
"""
import ctypes as C
import enum

import numpy as np

from . import _ffi as F
from ._ffi import SdrError, check, lib


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return int(x)


def _stream_ptr(stream):
    if stream is None:
        return None
    h = stream.cuda_stream if hasattr(stream, "cuda_stream") else int(stream)
    # NULL means "create your own stream" in the C ABI; the legacy default stream is cudaStreamLegacy (0x1)
    return h if h else 1


def device_count():
    return lib().sdr_device_count()


def device_info(dev=0):
    buf = C.create_string_buffer(256)
    check(lib().sdr_device_info(dev, buf, 256), "sdr_device_info")
    return buf.value.decode()


def kernel_launch_count():
    return int(lib().sdr_kernel_launch_count())


def unpack_u8iq(iq, device=0):
    """RtlTcpSignal::next over a whole buffer (src/rtltcp.rs:158-164)."""
    iq = np.ascontiguousarray(iq, np.uint8)
    n = iq.size // 2
    out = np.empty(n, np.complex64)
    check(lib().sdr_unpack_u8iq(iq.ctypes.data, n, out.ctypes.data, device), "sdr_unpack_u8iq")
    return out


def unpack_u8iq_dev(d_iq, n, d_out, device=0, stream=None):
    """device-resident unpack: d_iq 2n bytes, d_out n complex64, asynchronous on `stream`"""
    check(lib().sdr_unpack_u8iq_dev(_ptr(d_iq), n, _ptr(d_out), device, _stream_ptr(stream)), "sdr_unpack_u8iq_dev")


def decimate_wait(rate_in, rate_out):
    return lib().sdr_decimate_wait(rate_in, rate_out)


def duration_samples(rate, duration):
    return lib().sdr_duration_samples(rate, duration)


def block_samples(size, rate):
    return lib().sdr_block_samples(size, rate)


_FMT_OF = {"u8iq": F.FMT_U8IQ, "c64": F.FMT_C64, "f32": F.FMT_F32}
_IN_DTYPE = {F.FMT_U8IQ: np.uint8, F.FMT_C64: np.complex64, F.FMT_F32: np.float32}


class _Handle:
    """Owner of one C handle of the ABI family sdr_<_abi>_*: create, clone, reset and destroy."""
    _abi = None
    h = None

    def _fn(self, verb):
        return getattr(lib(), "sdr_%s_%s" % (self._abi, verb))

    def _create(self, cfg):
        err = C.c_int(0)
        self.h = self._fn("create")(C.byref(cfg), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_%s_create" % self._abi)

    def _adopt(self, h):
        """a copy of this object that owns handle h"""
        other = object.__new__(type(self))
        other.__dict__.update(self.__dict__)
        other.h = h
        return other

    def clone(self):
        err = C.c_int(0)
        h = self._fn("clone")(self.h, C.byref(err))
        if not h:
            raise SdrError(err.value, "sdr_%s_clone" % self._abi)
        return self._adopt(h)

    def reset(self):
        check(self._fn("reset")(self.h), "sdr_%s_reset" % self._abi)

    def close(self):
        if self.h:
            self._fn("destroy")(self.h)
            self.h = None

    def __del__(self):
        self.close()


class Fir(_Handle):
    """filter::Fir<C,A> with the signal::Filter (+ optional signal::Decimate) adaptor behaviour:
    a stateful stream filter.  taps float32 -> Fir<f32,A>; complex64 -> Fir<Complex<f32>,Complex<f32>>."""

    _abi = "fir"

    def __init__(self, taps, input_format="c64", decimation=1, n_channels=1, strict=False, device=0,
                 stream=None, flags=0):
        taps = np.asarray(taps)
        self.taps_complex = int(np.iscomplexobj(taps))
        self._taps = np.ascontiguousarray(taps, np.complex64 if self.taps_complex else np.float32)
        self.fmt = _FMT_OF[input_format] if isinstance(input_format, str) else int(input_format)
        self.decimation = int(decimation)
        self.n_channels = int(n_channels)
        self.device = device
        flags = int(flags) | (F.FIR_STRICT_ORDER if strict else 0)
        cfg = F.FirConfig(self._taps.ctypes.data, self._taps.size, self.taps_complex, self.fmt, self.decimation,
                          self.n_channels, flags, device, _stream_ptr(stream))
        self._create(cfg)

    @property
    def out_dtype(self):
        return np.float32 if self.fmt == F.FMT_F32 else np.complex64

    def output_count(self, n_in):
        return lib().sdr_fir_output_count(self.h, n_in)

    def process(self, x):
        """x: [n] or [n_channels, n] (u8 input: trailing dim 2n bytes).  Returns outputs for this block."""
        x = np.ascontiguousarray(x, _IN_DTYPE[self.fmt])
        per = 2 if self.fmt == F.FMT_U8IQ else 1
        rows = x.reshape(self.n_channels, -1)
        n_in = rows.shape[1] // per
        n_out = self.output_count(n_in)
        out = np.empty((self.n_channels, n_out), self.out_dtype)
        used, got = C.c_size_t(0), C.c_size_t(0)
        check(lib().sdr_fir_process(self.h, rows.ctypes.data, n_in, n_in, out.ctypes.data, n_out, n_out,
                                    C.byref(used), C.byref(got)), "sdr_fir_process")
        assert got.value == n_out and (used.value == n_in or n_in == 0)
        return out[0] if (self.n_channels == 1 and x.ndim <= 1) else out

    def process_dev(self, d_in, n_in, d_out, out_cap, in_stride=None, out_stride=None):
        used, got = C.c_size_t(0), C.c_size_t(0)
        check(lib().sdr_fir_process_dev(self.h, _ptr(d_in), n_in, in_stride or n_in, _ptr(d_out), out_cap,
                                        out_stride or out_cap, C.byref(used), C.byref(got)), "sdr_fir_process_dev")
        return got.value

    @property
    def last_path(self):
        return lib().sdr_fir_last_path(self.h)



class FftPlan:
    """Batched forward FFT with the post-processing of fft::fft (src/fft.rs:14-26) selectable by flags."""

    def __init__(self, n, input_format="c64", shift=False, norm=False, rfft=False, device=0, stream=None):
        self.n = int(n)
        self.fmt = _FMT_OF[input_format] if isinstance(input_format, str) else int(input_format)
        self.flags = (F.FFT_SHIFT if shift else 0) | (F.FFT_NORM if norm else 0) | (F.FFT_RFFT if rfft else 0)
        cfg = F.FftConfig(self.n, self.fmt, self.flags, device, _stream_ptr(stream))
        err = C.c_int(0)
        self.h = lib().sdr_fft_create(C.byref(cfg), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_fft_create")
        self.out_len = lib().sdr_fft_output_len(self.h)

    def exec(self, x):
        x = np.ascontiguousarray(x, _IN_DTYPE[self.fmt])
        per = 2 if self.fmt == F.FMT_U8IQ else 1
        batches = x.size // (per * self.n)
        out = np.empty((batches, self.out_len), np.complex64)
        check(lib().sdr_fft_exec(self.h, x.ctypes.data, batches, out.ctypes.data), "sdr_fft_exec")
        return out

    def exec_dev(self, d_in, batches, d_out):
        check(lib().sdr_fft_exec_dev(self.h, _ptr(d_in), batches, _ptr(d_out)), "sdr_fft_exec_dev")

    def close(self):
        if getattr(self, "h", None):
            lib().sdr_fft_destroy(self.h)
            self.h = None

    __del__ = close


def fft_labels(n, rate, rfft=False):
    out = np.empty(n - n // 2 if rfft else n, np.float32)
    check(lib().sdr_fft_labels(n, rate, int(rfft), out.ctypes.data), "sdr_fft_labels")
    return out


def fft(samples, rate=1.0, device=0):
    """fft::fft (src/fft.rs:3-28): one transform over the whole finite signal.
    Returns (labels f32[N], values complex64[N]) -- the reference's Vec<(f32, Complex<f32>)> unzipped."""
    x = np.ascontiguousarray(samples, np.complex64)
    if x.size == 0:
        return np.empty(0, np.float32), np.empty(0, np.complex64)
    plan = FftPlan(x.size, "c64", shift=True, norm=True, device=device)
    vals = plan.exec(x)[0]
    plan.close()
    return fft_labels(x.size, rate), vals


def rfft(samples, rate=1.0, device=0):
    """fft::rfft (src/fft.rs:30-37)."""
    x = np.ascontiguousarray(samples, np.float32)
    if x.size == 0:
        return np.empty(0, np.float32), np.empty(0, np.complex64)
    plan = FftPlan(x.size, "f32", shift=True, norm=True, rfft=True, device=device)
    vals = plan.exec(x)[0]
    plan.close()
    return fft_labels(x.size, rate, rfft=True), vals


class BiquadD:
    """filter::BiquadD (src/filter/biquad.rs:74-81) and filter::Identity, as (kind, p0, p1)."""

    def __init__(self, kind, p0=0.0, p1=0.0):
        self.kind, self.p0, self.p1 = kind, p0, p1

    @staticmethod
    def LowPass(freq, q): return BiquadD(F.BQ_LOWPASS, freq, q)
    @staticmethod
    def HighPass(freq, q): return BiquadD(F.BQ_HIGHPASS, freq, q)
    @staticmethod
    def BandPass(freq, q): return BiquadD(F.BQ_BANDPASS, freq, q)
    @staticmethod
    def Notch(freq, q): return BiquadD(F.BQ_NOTCH, freq, q)
    @staticmethod
    def Lr(decayrate): return BiquadD(F.BQ_LR, decayrate, 0.0)
    @staticmethod
    def Identity(): return BiquadD(F.BQ_IDENTITY)

    def _c(self):
        return F.BiquadDesign(self.kind, self.p0, self.p1)

    def coefficients(self, rate):
        out = np.empty(5, np.float32)
        d = self._c()
        check(lib().sdr_biquad_design(C.byref(d), rate, out.ctypes.data), "sdr_biquad_design")
        return out


Identity = BiquadD.Identity


class Biquad(_Handle):
    """filter::Biquad<f32, A> as a stream filter (biquad.rs:40-56): n_streams independent streams of f32 or
    Complex<f32> samples; designs = one BiquadD shared by all streams, or one per stream."""

    _abi = "biquad"

    def __init__(self, designs, rate, n_streams=1, complex_samples=False, device=0, stream=None):
        if isinstance(designs, BiquadD):
            designs = [designs]
        self.n_streams, self.complex_samples = int(n_streams), bool(complex_samples)
        arr = (F.BiquadDesign * len(designs))(*[d._c() for d in designs])
        self._arr = arr
        cfg = F.BiquadConfig(C.cast(arr, C.c_void_p), len(designs), self.n_streams, rate, int(self.complex_samples),
                             device, _stream_ptr(stream))
        self._create(cfg)

    def process(self, x):
        dt = np.complex64 if self.complex_samples else np.float32
        x = np.ascontiguousarray(x, dt)
        rows = x.reshape(self.n_streams, -1)
        n = rows.shape[1]
        out = np.empty_like(rows)
        check(lib().sdr_biquad_process(self.h, rows.ctypes.data, n, n, out.ctypes.data, n), "sdr_biquad_process")
        return out[0] if x.ndim <= 1 else out

    def process_dev(self, d_in, n, d_out, in_stride=None, out_stride=None):
        check(lib().sdr_biquad_process_dev(self.h, _ptr(d_in), n, in_stride or n, _ptr(d_out), out_stride or n),
              "sdr_biquad_process_dev")



class PllDesign:
    """filter::PllDesign::new(reference, gain, loopfilter, outputfilter, lockfilter) (pll.rs:26-36)."""

    def __init__(self, reference, gain, loopfilter, outputfilter, lockfilter):
        self.reference, self.gain = reference, gain
        self.loopfilter, self.outputfilter, self.lockfilter = loopfilter, outputfilter, lockfilter

    def _c(self):
        return F.PllDesign(self.reference, self.gain, self.loopfilter._c(), self.outputfilter._c(), self.lockfilter._c())

    def design(self, rate, n_streams=1, **kw):
        return PllBatch([self], n_streams, rate, **kw)


class PllBatch(_Handle):
    """n_streams independent filter::Pll instances (pll.rs:13-85)."""

    _abi = "pll"

    def __init__(self, designs, n_streams, rate, fast_math=True, device=0, stream=None, general=False):
        self.n_streams = int(n_streams)
        arr = (F.PllDesign * len(designs))(*[d._c() for d in designs])
        self._arr = arr
        cfg = F.PllConfig(C.cast(arr, C.c_void_p), len(designs), self.n_streams, rate,
                          (0 if fast_math else F.PLL_F64_MATH) | (F.PLL_GENERAL_KERNEL if general else 0), device,
                          _stream_ptr(stream))
        self._cfg = cfg
        self._create(cfg)

    def process(self, x):
        """x: complex64 [n] or [n_streams, n] -> (out f32, locked u8) of the same shape."""
        x = np.ascontiguousarray(x, np.complex64)
        rows = x.reshape(self.n_streams, -1)
        n = rows.shape[1]
        out = np.empty((self.n_streams, n), np.float32)
        locked = np.empty((self.n_streams, n), np.uint8)
        check(lib().sdr_pll_process(self.h, rows.ctypes.data, n, n, out.ctypes.data, locked.ctypes.data, n),
              "sdr_pll_process")
        if x.ndim <= 1:
            return out[0], locked[0]
        return out, locked

    def process_dev(self, d_in, n, d_out, d_locked, in_stride=None, out_stride=None):
        check(lib().sdr_pll_process_dev(self.h, _ptr(d_in), n, in_stride or n, _ptr(d_out), _ptr(d_locked),
                                        out_stride or n), "sdr_pll_process_dev")

    def stereo_decode(self, v):
        """the (mono, diff) closure of src/main.rs:62-71 around this (pilot) Pll: v f32 [n] or [n_streams, n] ->
        float32 [..., n, 2]"""
        v = np.ascontiguousarray(v, np.float32)
        rows = v.reshape(self.n_streams, -1)
        n = rows.shape[1]
        out = np.empty((self.n_streams, n, 2), np.float32)
        check(lib().sdr_pll_stereo_decode(self.h, rows.ctypes.data, n, n, out.ctypes.data, n), "sdr_pll_stereo_decode")
        return out[0] if v.ndim <= 1 else out

    def stereo_decode_dev(self, d_v, n, d_out, in_stride=None, out_stride=None):
        check(lib().sdr_pll_stereo_decode_dev(self.h, _ptr(d_v), n, in_stride or n, _ptr(d_out), out_stride or n),
              "sdr_pll_stereo_decode_dev")

    def state(self, idx=0):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        check(lib().sdr_pll_get_state(self.h, idx, C.byref(a), C.byref(b), C.byref(c)), "sdr_pll_get_state")
        return a.value, complex(b.value, c.value)



class WindowFft:
    """signal.window(duration).decimate(fps).map(fft::fft) of examples/live.rs:30-39: one spectrum per kept sliding
    window.  window = duration_samples(rate, duration), hop = decimate_wait(rate, fps)."""

    def __init__(self, window, hop, fmt="c64", shift=True, norm=True, device=0, stream=None):
        self.fmt = {"u8iq": F.FMT_U8IQ, "c64": F.FMT_C64}[fmt]
        flags = (F.FFT_SHIFT if shift else 0) | (F.FFT_NORM if norm else 0)
        cfg = F.WindowFftConfig(int(window), int(hop), self.fmt, flags, device, _stream_ptr(stream))
        err = C.c_int(0)
        self.h = lib().sdr_window_fft_create(C.byref(cfg), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_window_fft_create")
        self.window = int(window)

    def output_count(self, n_in):
        return lib().sdr_window_fft_output_count(self.h, n_in)

    def process(self, x):
        """x: uint8 [2n] (u8iq) or complex64 [n] -> complex64 [n_windows, window]"""
        if self.fmt == F.FMT_U8IQ:
            x = np.ascontiguousarray(x, np.uint8)
            n = x.size // 2
        else:
            x = np.ascontiguousarray(x, np.complex64)
            n = x.size
        nw = self.output_count(n)
        out = np.empty((max(nw, 1), self.window), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_window_fft_process(self.h, x.ctypes.data if n else None, n, out.ctypes.data, max(nw, 1),
                                           C.byref(got)), "sdr_window_fft_process")
        return out[:got.value]

    def process_dev(self, d_in, n, d_out, out_cap):
        got = C.c_size_t(0)
        check(lib().sdr_window_fft_process_dev(self.h, _ptr(d_in), n, _ptr(d_out), out_cap, C.byref(got)),
              "sdr_window_fft_process_dev")
        return got.value

    def reset(self):
        check(lib().sdr_window_fft_reset(self.h), "sdr_window_fft_reset")

    def close(self):
        if getattr(self, "h", None):
            lib().sdr_window_fft_destroy(self.h)
            self.h = None

    __del__ = close


class Pfb(_Handle):
    """Polyphase filter bank: one wideband stream -> n_channels channels decimated by `decimation`.  Channel k is
    Fir(h * exp(+2j pi k n / M)) followed by Decimate(D); channel k is centred on k * rate / M.  shift=True orders the
    channels like fft::fft's shift (row i = channel (i - M/2) mod M); channel_major=True returns [M, frames] instead of
    [frames, M].  general=True forces the general front-end kernel (same bits)."""

    _abi = "pfb"

    def __init__(self, taps, n_channels, decimation, input_format="c64", shift=False, channel_major=False,
                 general=False, device=0, stream=None):
        self._taps = np.ascontiguousarray(taps, np.float32)
        self.n_channels = int(n_channels)
        self.decimation = int(decimation)
        self.fmt = _FMT_OF[input_format] if isinstance(input_format, str) else int(input_format)
        self.channel_major = bool(channel_major)
        flags = (F.PFB_SHIFT if shift else 0) | (F.PFB_CHANNEL_MAJOR if channel_major else 0) | \
            (F.PFB_GENERAL_KERNEL if general else 0)
        cfg = F.PfbConfig(self._taps.ctypes.data, self._taps.size, self.n_channels, self.decimation, self.fmt, flags,
                          device, _stream_ptr(stream))
        self._create(cfg)

    def output_count(self, n_in):
        return lib().sdr_pfb_output_count(self.h, n_in)

    def process(self, x):
        """x: uint8 [2n] (u8iq) or complex64 [n] -> complex64 [frames, M] (or [M, frames] when channel-major)"""
        if self.fmt == F.FMT_U8IQ:
            x = np.ascontiguousarray(x, np.uint8)
            n = x.size // 2
        else:
            x = np.ascontiguousarray(x, np.complex64)
            n = x.size
        nf = self.output_count(n)
        M = self.n_channels
        cap = max(nf, 1)
        out = np.empty((M, cap) if self.channel_major else (cap, M), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_pfb_process(self.h, x.ctypes.data if n else None, n, out.ctypes.data, cap,
                                    cap if self.channel_major else M, C.byref(got)), "sdr_pfb_process")
        return out[:, :got.value] if self.channel_major else out[:got.value]

    def process_dev(self, d_in, n_in, d_out, out_cap, out_stride=None):
        """device-resident: d_in n_in samples, d_out frame-major (stride out_stride >= M) or channel-major (M rows of
        out_stride >= frames); asynchronous on the handle's stream.  Returns the frames written."""
        if out_stride is None:
            out_stride = out_cap if self.channel_major else self.n_channels
        got = C.c_size_t(0)
        check(lib().sdr_pfb_process_dev(self.h, _ptr(d_in), n_in, _ptr(d_out), out_cap, out_stride, C.byref(got)),
              "sdr_pfb_process_dev")
        return got.value



def ddc_phase_increment(freq, rate):
    """the 64-bit NCO increment of a channel centred on `freq` (Hz) in a stream of `rate` samples/s
    (sdr_ddc_phase_increment: nu = freq / rate folded into [-1/2, 1/2], rounded to nu * 2^64; negative = two's complement)"""
    return int(lib().sdr_ddc_phase_increment(float(freq), float(rate)))


class Pfs(_Handle):
    """Polyphase synthesis filter bank, the inverse of Pfb: frames of n_channels channel samples -> one stream at
    `interpolation` (D) samples per frame.  Channel k is zero-stuffed by D (sample m at index (m+1) D - 1), filtered by
    Fir(f * exp(+2j pi k n / M)) and summed over k; frame m releases outputs [m D, (m+1) D).  There is no scale: for
    unit round-trip gain f carries a factor D.  shift=True / channel_major=True take the layouts Pfb writes with the
    same flags ([frames, M] with row i = channel (i - M/2) mod M, or [M, frames]).  general=True forces the general
    back-end kernel (same bits)."""

    _abi = "pfs"

    def __init__(self, taps, n_channels, interpolation, shift=False, channel_major=False, general=False, device=0,
                 stream=None):
        self._taps = np.ascontiguousarray(taps, np.float32)
        self.n_channels = int(n_channels)
        self.interpolation = int(interpolation)
        self.channel_major = bool(channel_major)
        flags = (F.PFS_SHIFT if shift else 0) | (F.PFS_CHANNEL_MAJOR if channel_major else 0) | \
            (F.PFS_GENERAL_KERNEL if general else 0)
        cfg = F.PfsConfig(self._taps.ctypes.data, self._taps.size, self.n_channels, self.interpolation, flags, device,
                          _stream_ptr(stream))
        self._create(cfg)

    def output_count(self, n_frames):
        return lib().sdr_pfs_output_count(self.h, n_frames)

    def process(self, frames):
        """frames: complex64 [n, M] (or [M, n] when channel-major) -> complex64 [n * D]"""
        y = np.ascontiguousarray(frames, np.complex64)
        M = self.n_channels
        if y.ndim != 2 or y.shape[0 if self.channel_major else 1] != M:
            raise ValueError("frames must be [M, n] (channel-major) or [n, M] with M = %d" % M)
        n = y.shape[1] if self.channel_major else y.shape[0]
        cnt = self.output_count(n)
        out = np.empty(max(cnt, 1), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_pfs_process(self.h, y.ctypes.data if n else None, n, n if self.channel_major else M,
                                    out.ctypes.data, cnt, C.byref(got)), "sdr_pfs_process")
        return out[:got.value]

    def process_dev(self, d_in, n_frames, d_out, out_cap, in_stride=None):
        """device-resident: d_in n_frames frames, frame-major (stride in_stride >= M) or channel-major (M rows of
        in_stride >= n_frames); d_out out_cap samples; asynchronous on the handle's stream.  Returns the samples
        written (n_frames * D)."""
        if in_stride is None:
            in_stride = n_frames if self.channel_major else self.n_channels
        got = C.c_size_t(0)
        check(lib().sdr_pfs_process_dev(self.h, _ptr(d_in), n_frames, in_stride, _ptr(d_out), out_cap, C.byref(got)),
              "sdr_pfs_process_dev")
        return got.value



class Ddc(_Handle):
    """Digital down-converter bank: channel k of one IQ stream is mixed down by freqs[k] (a 64-bit NCO), filtered by its
    real taps (taps 1-D: shared; [C, L]: one row per channel) and decimated by `decimation`:
    y_k[m] = sum_j h_k[j] x[N - j] e^{-2 pi i phi_k(N - j)}, N = (m + 1) D - 1.  first_sample = absolute stream index of
    the first input (places the NCO phase only).  process returns complex64 [C, outputs] (channel-major rows).
    general=True forces the CUDA-core kernel."""

    _abi = "ddc"

    def __init__(self, taps, freqs, rate, decimation, input_format="u8iq", first_sample=0, general=False, device=0,
                 stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        self._taps = t
        self.phase_inc = np.array([ddc_phase_increment(f, rate) for f in np.atleast_1d(freqs)], np.uint64)
        self.n_channels = int(self.phase_inc.size)
        self.decimation = int(decimation)
        self.fmt = _FMT_OF[input_format] if isinstance(input_format, str) else int(input_format)
        cfg = F.DdcConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phase_inc.ctypes.data,
                          self.n_channels, self.decimation, int(first_sample), self.fmt,
                          F.DDC_GENERAL_KERNEL if general else 0, device, _stream_ptr(stream))
        self._create(cfg)

    def output_count(self, n_in):
        return lib().sdr_ddc_output_count(self.h, n_in)

    @property
    def last_path(self):
        """path of the last call that produced outputs: 0 none, 1 CUDA-core kernel, 2 tcgen05 kernel"""
        return lib().sdr_ddc_last_path(self.h)

    def process(self, x):
        """x: uint8 [2n] (u8iq) or complex64 [n] -> complex64 [C, outputs]"""
        if self.fmt == F.FMT_U8IQ:
            x = np.ascontiguousarray(x, np.uint8)
            n = x.size // 2
        else:
            x = np.ascontiguousarray(x, np.complex64)
            n = x.size
        cap = max(self.output_count(n), 1)
        out = np.empty((self.n_channels, cap), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_ddc_process(self.h, x.ctypes.data if n else None, n, out.ctypes.data, cap, cap, C.byref(got)),
              "sdr_ddc_process")
        return out[:, :got.value]

    def process_dev(self, d_in, n_in, d_out, out_cap, out_stride=None):
        """device-resident: d_in n_in samples, d_out C rows of out_stride (default out_cap) complex64; asynchronous on
        the handle's stream.  Returns the outputs written per channel."""
        got = C.c_size_t(0)
        check(lib().sdr_ddc_process_dev(self.h, _ptr(d_in), n_in, _ptr(d_out), out_cap,
                                        out_cap if out_stride is None else out_stride, C.byref(got)),
              "sdr_ddc_process_dev")
        return got.value



class Duc(_Handle):
    """Digital up-converter bank, the transpose of Ddc: channel k (row k of a [C, n] complex64 array) is zero-stuffed
    by `interpolation` (I; sample m at index (m+1) I - 1), filtered by its real taps (1-D: shared; [C, L]: one row
    per channel), mixed UP by freqs[k] (a 64-bit NCO) and all channels are summed:
    x[n] = sum_k u_k[n] e^{+2 pi i phi_k(first_sample + n)}.  first_sample = absolute stream index of the first
    OUTPUT (places the NCO phase only).  Frame m releases outputs [m I, (m+1) I).  There is no scale: for unit
    round-trip gain after Ddc the taps carry the factor I, and first_sample is the Ddc's minus the cascade's delay."""

    _abi = "duc"

    def __init__(self, taps, freqs, rate, interpolation, first_sample=0, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        self._taps = t
        self.phase_inc = np.array([ddc_phase_increment(f, rate) for f in np.atleast_1d(freqs)], np.uint64)
        self.n_channels = int(self.phase_inc.size)
        self.interpolation = int(interpolation)
        cfg = F.DucConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phase_inc.ctypes.data,
                          self.n_channels, self.interpolation, int(first_sample) % (1 << 64), 0, device,
                          _stream_ptr(stream))
        self._create(cfg)

    def output_count(self, n_frames):
        return lib().sdr_duc_output_count(self.h, n_frames)

    def process(self, y):
        """y: complex64 [C, n] (row k = channel k) -> complex64 [n * I]"""
        y = np.ascontiguousarray(y, np.complex64)
        if y.ndim == 1 and self.n_channels == 1:
            y = y[None]
        if y.ndim != 2 or y.shape[0] != self.n_channels:
            raise ValueError("y must be [C, n] with C = %d" % self.n_channels)
        n = y.shape[1]
        cnt = self.output_count(n)
        out = np.empty(max(cnt, 1), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_duc_process(self.h, y.ctypes.data if n else None, n, n, out.ctypes.data, cnt, C.byref(got)),
              "sdr_duc_process")
        return out[:got.value]

    def process_dev(self, d_in, n_frames, d_out, out_cap, in_stride=None):
        """device-resident: d_in C rows of in_stride (default n_frames) complex64, n_frames each; d_out out_cap samples;
        asynchronous on the handle's stream.  Returns the samples written (n_frames * I)."""
        got = C.c_size_t(0)
        check(lib().sdr_duc_process_dev(self.h, _ptr(d_in), n_frames, n_frames if in_stride is None else in_stride,
                                        _ptr(d_out), out_cap, C.byref(got)), "sdr_duc_process_dev")
        return got.value



class Psd(_Handle):
    """Averaged power spectra (sdr_psd): window(n) -> decimate(hop) -> map(fft::fft) -> |.|^2 -> mean of `average`
    frames.  Frame j holds the n samples ending at input sample (j + 1) * hop - 1 (x[<0] = 0), tapered by `window`
    (n real values, None = rectangular); spectrum g is the mean of |X_j|^2 over frames g*average .. g*average +
    average - 1, as float32 rows of n bins.  shift / norm as for FftPlan (norm scales the rows by 1/n).  average=1 is a
    waterfall.  general=True forces the plan + slab path (path 1) where the fused 1024-point kernel (path 2) would run."""

    _abi = "psd"

    def __init__(self, n, hop, average, window=None, fmt="u8iq", shift=True, norm=True, general=False, device=0,
                 stream=None):
        self.n, self.hop, self.average = int(n), int(hop), int(average)
        self.fmt = _FMT_OF[fmt] if isinstance(fmt, str) else int(fmt)
        self._window = None if window is None else np.ascontiguousarray(window, np.float32)
        if self._window is not None and self._window.size != self.n:
            raise ValueError("window must hold n taper values")
        flags = (F.PSD_SHIFT if shift else 0) | (F.PSD_NORM if norm else 0) | (F.PSD_GENERAL_KERNEL if general else 0)
        cfg = F.PsdConfig(self.n, self.hop, self.average, None if self._window is None else self._window.ctypes.data,
                          self.fmt, flags, device, _stream_ptr(stream))
        self._create(cfg)

    def output_count(self, n_in):
        return lib().sdr_psd_output_count(self.h, n_in)

    @property
    def last_path(self):
        """path of the last call that ran frames: 0 none, 1 plan + slab, 2 fused 1024-point kernel"""
        return lib().sdr_psd_last_path(self.h)

    def process(self, x):
        """x: uint8 [2m] (u8iq) or complex64 [m] -> float32 [spectra, n]"""
        if self.fmt == F.FMT_U8IQ:
            x = np.ascontiguousarray(x, np.uint8)
            m = x.size // 2
        else:
            x = np.ascontiguousarray(x, np.complex64)
            m = x.size
        cap = max(self.output_count(m), 1)
        out = np.empty((cap, self.n), np.float32)
        got = C.c_size_t(0)
        check(lib().sdr_psd_process(self.h, x.ctypes.data if m else None, m, out.ctypes.data, cap, self.n,
                                    C.byref(got)), "sdr_psd_process")
        return out[:got.value]

    def process_dev(self, d_in, n_in, d_out, out_cap, out_stride=None):
        """device-resident: d_in n_in samples, d_out rows of out_stride (default n) float32; asynchronous on the
        handle's stream.  Returns the spectra written."""
        got = C.c_size_t(0)
        check(lib().sdr_psd_process_dev(self.h, _ptr(d_in), n_in, _ptr(d_out), out_cap,
                                        self.n if out_stride is None else out_stride, C.byref(got)),
              "sdr_psd_process_dev")
        return got.value



def fcfb_geometry(n_taps, decimations):
    """(N, P): the transform size and hop sdr_fcfb uses for n_taps taps and these per-channel decimations"""
    d = np.ascontiguousarray(np.atleast_1d(decimations), np.uintp)
    n, p = C.c_size_t(0), C.c_size_t(0)
    check(lib().sdr_fcfb_geometry(int(n_taps), d.ctypes.data, d.size, C.byref(n), C.byref(p)), "sdr_fcfb_geometry")
    return n.value, p.value


class Fcfb(_Handle):
    """Fast-convolution channel bank (sdr_fcfb): channel k of one IQ stream is mixed down by freqs[k] (a 64-bit NCO),
    filtered by its real taps (taps 1-D: shared; [C, L]: one row per channel) and decimated by decimation[k] (one value
    or one per channel) -- sdr_ddc's channel with its own D -- computed by overlap-save on blocks of N inputs.  Outputs
    are released per block of P inputs (see geometry); process returns a list of C complex64 arrays.  To drain a finite
    stream feed N zeros and drop the outputs past its end."""

    _abi = "fcfb"

    def __init__(self, taps, freqs, rate, decimation, input_format="u8iq", first_sample=0, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        self._taps = t
        self.phase_inc = np.array([ddc_phase_increment(f, rate) for f in np.atleast_1d(freqs)], np.uint64)
        self.n_channels = int(self.phase_inc.size)
        d = np.atleast_1d(np.asarray(decimation, np.int64))
        if d.size == 1:
            d = np.repeat(d, self.n_channels)
        if d.size != self.n_channels or (d < 1).any():
            raise ValueError("decimation: one value >= 1, or one per channel")
        self.decimation = np.ascontiguousarray(d, np.uintp)
        self.fmt = _FMT_OF[input_format] if isinstance(input_format, str) else int(input_format)
        cfg = F.FcfbConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phase_inc.ctypes.data,
                           self.decimation.ctypes.data, self.n_channels, int(first_sample), self.fmt, device,
                           _stream_ptr(stream))
        self._create(cfg)

    @property
    def geometry(self):
        """(N, P): transform size and hop (inputs per block)"""
        return fcfb_geometry(self._taps.shape[-1], self.decimation)

    def output_count(self, n_in):
        """outputs per channel (numpy array of C) of the blocks that the next n_in inputs complete"""
        cnt = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fcfb_output_count(self.h, n_in, cnt.ctypes.data), "sdr_fcfb_output_count")
        return cnt.astype(np.int64)

    def process(self, x):
        """x: uint8 [2n] (u8iq) or complex64 [n] -> list of C complex64 arrays"""
        if self.fmt == F.FMT_U8IQ:
            x = np.ascontiguousarray(x, np.uint8)
            n = x.size // 2
        else:
            x = np.ascontiguousarray(x, np.complex64)
            n = x.size
        cap = max(int(self.output_count(n).max()), 1)
        out = np.empty((self.n_channels, cap), np.complex64)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fcfb_process(self.h, x.ctypes.data if n else None, n, out.ctypes.data, cap, cap,
                                     got.ctypes.data), "sdr_fcfb_process")
        return [out[k, :int(got[k])] for k in range(self.n_channels)]

    def process_dev(self, d_in, n_in, d_out, out_cap, out_stride=None):
        """device-resident: d_in n_in samples, d_out C rows of out_stride (default out_cap) complex64; asynchronous on
        the handle's stream.  Returns the outputs written per channel (numpy array of C)."""
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fcfb_process_dev(self.h, _ptr(d_in), n_in, _ptr(d_out), out_cap,
                                         out_cap if out_stride is None else out_stride, got.ctypes.data),
              "sdr_fcfb_process_dev")
        return got.astype(np.int64)



class Fcsb(_Handle):
    """Fast-convolution synthesis bank (sdr_fcsb), the inverse of Fcfb: channel k is zero-stuffed by interpolation[k]
    (I_k, one value or one per channel; frame m at index (m+1) I_k - 1), filtered by its real taps (1-D: shared;
    [C, L]: one row per channel), mixed UP by freqs[k] (a 64-bit NCO) and all channels are summed -- Duc's function
    with its own I per channel -- computed by overlap-save on Fcfb's geometry.  first_sample = absolute stream index of
    the first OUTPUT.  A call advances the handle by n_time output positions (a multiple of lcm(I_k)) and returns the
    outputs of the blocks it completes (see geometry); to drain a finite stream feed zero frames covering N positions
    and drop the outputs past its end.  There is no scale: the taps carry the factor I_k."""

    _abi = "fcsb"

    def __init__(self, taps, freqs, rate, interpolation, first_sample=0, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        self._taps = t
        self.phase_inc = np.array([ddc_phase_increment(f, rate) for f in np.atleast_1d(freqs)], np.uint64)
        self.n_channels = int(self.phase_inc.size)
        i = np.atleast_1d(np.asarray(interpolation, np.int64))
        if i.size == 1:
            i = np.repeat(i, self.n_channels)
        if i.size != self.n_channels or (i < 1).any():
            raise ValueError("interpolation: one value >= 1, or one per channel")
        self.interpolation = np.ascontiguousarray(i, np.uintp)
        self.lcm = int(np.lcm.reduce(i))
        cfg = F.FcsbConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phase_inc.ctypes.data,
                           self.interpolation.ctypes.data, self.n_channels, int(first_sample) % (1 << 64), device,
                           _stream_ptr(stream))
        self._create(cfg)

    @property
    def geometry(self):
        """(N, P): transform size and hop (output positions per block)"""
        return fcfb_geometry(self._taps.shape[-1], self.interpolation)

    def output_count(self, n_time):
        """outputs of the blocks that the next n_time output positions complete"""
        return lib().sdr_fcsb_output_count(self.h, n_time)

    def process(self, rows):
        """rows: C complex64 arrays (or a [C, n] array when every I_k is equal), row k of n_k frames with the same
        n_k I_k for every k -> complex64 [released outputs]"""
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n_time = rows[0].size * int(self.interpolation[0])
        if any(r.size * int(i) != n_time for r, i in zip(rows, self.interpolation)):
            raise ValueError("rows: n_k I_k must be equal for every channel")
        stride = max(max(r.size for r in rows), 1)
        y = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            y[k, :r.size] = r
        cnt = self.output_count(n_time)
        out = np.empty(max(cnt, 1), np.complex64)
        got = C.c_size_t(0)
        check(lib().sdr_fcsb_process(self.h, y.ctypes.data if n_time else None, n_time, stride, out.ctypes.data, cnt,
                                     C.byref(got)), "sdr_fcsb_process")
        return out[:got.value]

    def process_dev(self, d_in, n_time, d_out, out_cap, in_stride=None):
        """device-resident: d_in C rows of in_stride (default the longest row, n_time / min I_k) complex64, row k
        n_time / I_k frames; d_out out_cap samples; asynchronous on the handle's stream.  Returns the samples written."""
        stride = n_time // int(self.interpolation.min()) if in_stride is None else in_stride
        got = C.c_size_t(0)
        check(lib().sdr_fcsb_process_dev(self.h, _ptr(d_in), n_time, stride, _ptr(d_out), out_cap, C.byref(got)),
              "sdr_fcsb_process_dev")
        return got.value



class Rrb(_Handle):
    """Rational resampler bank (sdr_rrb), the textbook upfirdn per channel: channel k is zero-stuffed by
    interpolation[k] (I_k; frame m at index (m+1) I_k - 1), filtered by its real taps (1-D: shared; [C, L]: one row per
    channel) and decimated by decimation[k] (D_k; output r is sample (r+1) D_k - 1).  interpolation and decimation
    take one value or one per channel.  After n frames a channel has released floor(n I_k / D_k) outputs.  There is no
    scale: unit gain needs taps with DC gain I_k."""

    _abi = "rrb"

    def __init__(self, taps, interpolation, decimation, n_channels=None, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        i = np.atleast_1d(np.asarray(interpolation, np.int64))
        d = np.atleast_1d(np.asarray(decimation, np.int64))
        c = int(n_channels) if n_channels is not None else max(i.size, d.size, 1 if t.ndim == 1 else t.shape[0])
        i = np.repeat(i, c) if i.size == 1 else i
        d = np.repeat(d, c) if d.size == 1 else d
        if i.size != c or d.size != c or (i < 1).any() or (d < 1).any():
            raise ValueError("interpolation / decimation: one value >= 1, or one per channel")
        self._taps = t
        self.n_channels = c
        self.interpolation = np.ascontiguousarray(i, np.uintp)
        self.decimation = np.ascontiguousarray(d, np.uintp)
        cfg = F.RrbConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.interpolation.ctypes.data,
                          self.decimation.ctypes.data, c, device, _stream_ptr(stream))
        self._create(cfg)

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def output_count(self, n_in):
        """outputs per channel (numpy array of C) from the next n_in frames (an int, or one count per channel)"""
        n = self._counts(n_in)
        cnt = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_rrb_output_count(self.h, n.ctypes.data, cnt.ctypes.data), "sdr_rrb_output_count")
        return cnt.astype(np.int64)

    def process(self, rows):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> list of C complex64 arrays"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        y = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            y[k, :r.size] = r
        cnt = self.output_count(n)
        cap = max(int(cnt.max()), 1)
        out = np.empty((self.n_channels, cap), np.complex64)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_rrb_process(self.h, y.ctypes.data, n.ctypes.data, stride, out.ctypes.data, cap, cap,
                                    got.ctypes.data), "sdr_rrb_process")
        return [out[k, :int(got[k])] for k in range(self.n_channels)]

    def process_dev(self, d_in, n_in, in_stride, d_out, out_cap, out_stride):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) frames; d_out C rows
        of out_stride complex64, out_cap outputs each; asynchronous on the handle's stream.  Returns the outputs written
        per channel (numpy array of C)."""
        n = self._counts(n_in)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_rrb_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), out_cap, out_stride,
                                        got.ctypes.data), "sdr_rrb_process_dev")
        return got.astype(np.int64)



_ONE = 1 << 64  # one input frame in the units of Arb's steps and positions


def _arb_times(v, c, what):
    """ints in units of 2^-64 frames (one, or one per channel) -> ctypes array of c ArbTime"""
    v = [int(x) for x in (v if hasattr(v, "__len__") else [v])]
    v = v * c if len(v) == 1 else v
    if len(v) != c or any(x < 0 or x >> 128 for x in v):
        raise ValueError("%s: one value in [0, 2^128), or one per channel, in units of 2^-64 frames" % what)
    return (F.ArbTime * c)(*[F.ArbTime(x >> 64, x & (_ONE - 1)) for x in v])


def arb_step(rate_in, rate_out):
    """rate_in / rate_out rounded to the nearest 2^-64 (ties to even), as an int in units of 2^-64 frames"""
    t = F.ArbTime()
    check(lib().sdr_arb_step(float(rate_in), float(rate_out), C.byref(t)), "sdr_arb_step")
    return (t.whole << 64) | t.frac


class Arb(_Handle):
    """Arbitrary-ratio resampler bank (sdr_arb): channel k resampled by its own step sigma_k (input frames per output)
    on an exact time base, with real taps designed at `phases` (P, a power of two) times the input rate (1-D: shared;
    [C, L]: one row per channel), linearly interpolated between adjacent phases.  Output r sits at
    tau_k(r) = first_k + r sigma_k.  steps and first are Python ints in units of 2^-64 frames (arb_step converts a rate
    pair), one value or one per channel; first defaults to 0.  After n frames a channel has released
    #{r : tau(r) < n} outputs.  There is no scale: unit gain needs sum(taps) = P."""

    _abi = "arb"

    def __init__(self, taps, phases, steps, first=None, n_channels=None, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        ns = len(steps) if hasattr(steps, "__len__") else 1
        nf = len(first) if hasattr(first, "__len__") else 1
        c = int(n_channels) if n_channels is not None else max(ns, nf, 1 if t.ndim == 1 else t.shape[0])
        self._taps = t
        self.n_channels = c
        self.phases = int(phases)
        self._steps = _arb_times(steps, c, "steps")
        self._first = None if first is None else _arb_times(first, c, "first")
        cfg = F.ArbConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phases,
                          C.addressof(self._steps), None if self._first is None else C.addressof(self._first), c,
                          device, _stream_ptr(stream))
        self._create(cfg)

    def set_steps(self, steps):
        """new steps (ints in units of 2^-64, one or one per channel) from each channel's next unreleased output on"""
        s = _arb_times(steps, self.n_channels, "steps")
        check(lib().sdr_arb_set_steps(self.h, C.addressof(s)), "sdr_arb_set_steps")

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def output_count(self, n_in):
        """outputs per channel (numpy array of C) from the next n_in frames (an int, or one count per channel)"""
        n = self._counts(n_in)
        cnt = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_arb_output_count(self.h, n.ctypes.data, cnt.ctypes.data), "sdr_arb_output_count")
        return cnt.astype(np.int64)

    def process(self, rows):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> list of C complex64 arrays"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        y = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            y[k, :r.size] = r
        cnt = self.output_count(n)
        cap = max(int(cnt.max()), 1)
        out = np.empty((self.n_channels, cap), np.complex64)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_arb_process(self.h, y.ctypes.data, n.ctypes.data, stride, out.ctypes.data, cap, cap,
                                    got.ctypes.data), "sdr_arb_process")
        return [out[k, :int(got[k])] for k in range(self.n_channels)]

    def process_dev(self, d_in, n_in, in_stride, d_out, out_cap, out_stride):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) frames; d_out C rows
        of out_stride complex64, out_cap outputs each; asynchronous on the handle's stream.  Returns the outputs written
        per channel (numpy array of C)."""
        n = self._counts(n_in)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_arb_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), out_cap, out_stride,
                                        got.ctypes.data), "sdr_arb_process_dev")
        return got.astype(np.int64)


def tsync_loop_design(bn_t, zeta, ted_gain, period_frames):
    """(kp, ki) of the standard second-order loop, in frames per unit of detector output: noise bandwidth bn_t
    (normalised to the symbol rate), damping zeta, detector slope ted_gain (mean e per symbol period of timing error)"""
    kp, ki = C.c_float(), C.c_float()
    check(lib().sdr_tsync_loop_design(float(bn_t), float(zeta), float(ted_gain), float(period_frames), C.byref(kp),
                                      C.byref(ki)), "sdr_tsync_loop_design")
    return kp.value, ki.value


def _positions(a):
    """[n, 2] uint64 (whole, frac) -> list of Python ints in units of 2^-64 frames"""
    return [(int(w) << 64) | int(f) for w, f in a]


class Tsync(_Handle):
    """Symbol timing recovery bank (sdr_tsync): a Gardner loop per channel that steers sdr_arb's interpolator.  taps:
    the matched filter at `phases` (P, a power of two) times the input rate (1-D: shared; [C, L]: one row per channel);
    periods and first: Python ints in units of 2^-64 frames (arb_step(rate, symbol_rate) gives a period), one value or
    one per channel, first defaulting to 0; loops: one (kp, ki, err_max, max_dev) or one per channel.  process returns
    the symbols y_s, their exact positions tau_s and the detector outputs e_s; see include/sdr_b200.h for the
    recurrence."""

    _abi = "tsync"

    def __init__(self, taps, phases, periods, loops, first=None, n_channels=None, device=0, stream=None):
        t = np.ascontiguousarray(taps, np.float32)
        if t.ndim not in (1, 2):
            raise ValueError("taps must be 1-D (shared) or [channels, taps]")
        lp = [loops] if np.ndim(loops[0]) == 0 else list(loops)
        ns = len(periods) if hasattr(periods, "__len__") else 1
        nf = len(first) if hasattr(first, "__len__") else 1
        c = int(n_channels) if n_channels is not None else max(ns, nf, len(lp), 1 if t.ndim == 1 else t.shape[0])
        self._taps = t
        self.n_channels = c
        self.phases = int(phases)
        self._periods = _arb_times(periods, c, "periods")
        self._first = None if first is None else _arb_times(first, c, "first")
        self._loops = (F.TsyncLoop * len(lp))(*[F.TsyncLoop(*map(float, x)) for x in lp])
        cfg = F.TsyncConfig(t.ctypes.data, t.shape[-1], 1 if t.ndim == 1 else t.shape[0], self.phases,
                            C.addressof(self._periods), None if self._first is None else C.addressof(self._first),
                            C.addressof(self._loops), len(lp), c, device, _stream_ptr(stream))
        self._create(cfg)

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def max_output(self, n_in):
        """the most symbols per channel (numpy array of C) the next n_in frames (an int, or one per channel) release"""
        n = self._counts(n_in)
        cap = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_tsync_max_output(self.h, n.ctypes.data, cap.ctypes.data), "sdr_tsync_max_output")
        return cap.astype(np.int64)

    def state(self, k):
        """(next unreleased position as an int in units of 2^-64 frames, v in units of 2^-40 frames) of channel k"""
        t, v = F.ArbTime(), C.c_int64()
        check(lib().sdr_tsync_get_state(self.h, int(k), C.byref(t), C.byref(v)), "sdr_tsync_get_state")
        return (t.whole << 64) | t.frac, v.value

    def process(self, rows):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> (symbols, positions, errors): lists of C
        complex64 arrays, C lists of Python ints (units of 2^-64 frames) and C float32 arrays"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        y = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            y[k, :r.size] = r
        cap = max(int(self.max_output(n).max()), 1)
        sym = np.empty((self.n_channels, cap), np.complex64)
        pos = np.empty((self.n_channels, cap, 2), np.uint64)
        err = np.empty((self.n_channels, cap), np.float32)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_tsync_process(self.h, y.ctypes.data, n.ctypes.data, stride, sym.ctypes.data, pos.ctypes.data,
                                      err.ctypes.data, cap, cap, got.ctypes.data), "sdr_tsync_process")
        g = [int(x) for x in got]
        return ([sym[k, :g[k]] for k in range(self.n_channels)],
                [_positions(pos[k, :g[k]]) for k in range(self.n_channels)],
                [err[k, :g[k]] for k in range(self.n_channels)])

    def process_dev(self, d_in, n_in, in_stride, d_sym, out_cap, out_stride, d_pos=None, d_err=None):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) frames; d_sym C rows
        of out_stride complex64 (out_cap >= max_output); d_pos (int64 [C, out_stride, 2]: whole, frac) and d_err
        (float32 [C, out_stride]) may be None.  Returns the symbols written per channel (numpy array of C) once they
        are known, which synchronises the handle's stream."""
        n = self._counts(n_in)
        got = np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_tsync_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_sym), _ptr(d_pos),
                                          _ptr(d_err), out_cap, out_stride, got.ctypes.data), "sdr_tsync_process_dev")
        return got.astype(np.int64)


class Csync(_Handle):
    """Carrier recovery bank (sdr_csync): a decision-directed Costas loop per channel on an exact 64-bit phase.  loops:
    one (order, kp, ki, err_max, max_freq) or one per channel, order M in {2, 4, 8} (BPSK, QPSK, 8PSK), kp and ki in
    turns per unit of detector output (tsync_loop_design(bn_t, zeta, K_d, 1 / (2 pi))), max_freq in turns per symbol;
    phase (units of 2^-64 turn) and freq (units of 2^-40 turn per symbol): Python ints, one value or one per channel,
    defaulting to 0.  process returns the derotated symbols z_s, their phases phi_s and the detector outputs e_s; see
    include/sdr_b200.h for the recurrence."""

    _abi = "csync"

    def __init__(self, loops, n_channels=None, phase=None, freq=None, device=0, stream=None):
        lp = [loops] if np.ndim(loops[0]) == 0 else list(loops)
        npd = len(phase) if hasattr(phase, "__len__") else 1
        nfq = len(freq) if hasattr(freq, "__len__") else 1
        c = int(n_channels) if n_channels is not None else max(len(lp), npd, nfq)
        self.n_channels = c
        self._loops = (F.CsyncLoop * len(lp))(*[F.CsyncLoop(int(x[0]), *map(float, x[1:])) for x in lp])
        self._phase = None if phase is None else (C.c_uint64 * c)(*self._per_channel(phase, c, 0, 1 << 64, "phase"))
        self._freq = None if freq is None else (C.c_int64 * c)(*self._per_channel(freq, c, -(1 << 63), 1 << 63,
                                                                                  "freq"))
        cfg = F.CsyncConfig(C.addressof(self._loops), len(lp),
                            None if self._phase is None else C.addressof(self._phase),
                            None if self._freq is None else C.addressof(self._freq), c, device, _stream_ptr(stream))
        self._create(cfg)

    @staticmethod
    def _per_channel(v, c, lo, hi, what):
        v = [int(x) for x in (v if hasattr(v, "__len__") else [v])]
        v = v * c if len(v) == 1 else v
        if len(v) != c or any(x < lo or x >= hi for x in v):
            raise ValueError("%s: one value in [%d, %d), or one per channel" % (what, lo, hi))
        return v

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def state(self, k):
        """(phase in units of 2^-64 turn, freq in units of 2^-40 turn per symbol) of channel k's next symbol"""
        ph, fr = C.c_uint64(), C.c_int64()
        check(lib().sdr_csync_get_state(self.h, int(k), C.byref(ph), C.byref(fr)), "sdr_csync_get_state")
        return ph.value, fr.value

    def process(self, rows):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> (symbols, phases, errors): lists of C complex64,
        uint64 (units of 2^-64 turn) and float32 arrays, as long as the rows"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        y = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            y[k, :r.size] = r
        z = np.empty_like(y)
        ph = np.empty((self.n_channels, stride), np.uint64)
        err = np.empty((self.n_channels, stride), np.float32)
        check(lib().sdr_csync_process(self.h, y.ctypes.data, n.ctypes.data, stride, z.ctypes.data, ph.ctypes.data,
                                      err.ctypes.data, stride), "sdr_csync_process")
        g = [int(x) for x in n]
        return ([z[k, :g[k]] for k in range(self.n_channels)], [ph[k, :g[k]] for k in range(self.n_channels)],
                [err[k, :g[k]] for k in range(self.n_channels)])

    def process_dev(self, d_in, n_in, in_stride, d_out, out_stride, d_phase=None, d_err=None):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) symbols; d_out C rows
        of out_stride complex64 (may be d_in with the same stride); d_phase (int64 or uint64 [C, out_stride]) and d_err
        (float32 [C, out_stride]) may be None.  Asynchronous on the handle's stream: row k gets n_in[k] symbols."""
        n = self._counts(n_in)
        check(lib().sdr_csync_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), _ptr(d_phase),
                                          _ptr(d_err), out_stride), "sdr_csync_process_dev")


class Eq(_Handle):
    """Adaptive equalizer bank (sdr_eq): an n_taps-tap FIR per channel whose complex weights adapt by blind CMA and then
    decision-directed LMS.  adapt: one (order, mu, radius, err_max, cma_symbols) or one per channel, order M in
    {2, 4, 8} (the DD decisions: BPSK, QPSK, 8PSK at the radius), cma_symbols S: symbols s < S adapt by CMA, later ones
    by DD (None or 2**64 - 1: CMA only; 0: DD only).  taps: None (the centre spike), N complex taps shared, or [C, N];
    n_channels defaults to the number of adaptation or tap sets.  process returns the equalized symbols y_s and the
    errors e_s; see include/sdr_b200.h for the recurrence."""

    _abi = "eq"

    def __init__(self, n_taps, adapt, n_channels=None, taps=None, device=0, stream=None):
        ad = [adapt] if np.ndim(adapt[0]) == 0 else list(adapt)
        N = int(n_taps)
        t = None if taps is None else np.ascontiguousarray(np.asarray(taps, np.complex64).reshape(-1, N))
        c = int(n_channels) if n_channels is not None else max(len(ad), 1 if t is None else len(t))
        self.n_channels, self.n_taps = c, N

        def one(a):
            S = (1 << 64) - 1 if a[4] is None else int(a[4])
            return F.EqAdapt(int(a[0]), float(a[1]), float(a[2]), float(a[3]), S)
        self._adapt = (F.EqAdapt * len(ad))(*[one(a) for a in ad])
        self._taps = t
        cfg = F.EqConfig(N, None if t is None else t.ctypes.data, 0 if t is None else len(t), C.addressof(self._adapt),
                         len(ad), c, device, _stream_ptr(stream))
        self._create(cfg)

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def taps(self, k):
        """channel k's N complex64 taps for its next symbol"""
        w = np.empty(self.n_taps, np.complex64)
        check(lib().sdr_eq_get_taps(self.h, int(k), w.ctypes.data), "sdr_eq_get_taps")
        return w

    def process(self, rows):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> (y, e): lists of C complex64 arrays, as long as
        the rows"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        x = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            x[k, :r.size] = r
        y = np.empty_like(x)
        e = np.empty_like(x)
        check(lib().sdr_eq_process(self.h, x.ctypes.data, n.ctypes.data, stride, y.ctypes.data, e.ctypes.data,
                                   stride), "sdr_eq_process")
        g = [int(v) for v in n]
        return [y[k, :g[k]] for k in range(self.n_channels)], [e[k, :g[k]] for k in range(self.n_channels)]

    def process_dev(self, d_in, n_in, in_stride, d_out, out_stride, d_err=None):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) symbols; d_out C
        rows of out_stride complex64 (may be d_in with the same stride); d_err (complex64 [C, out_stride]) may be None.
        Asynchronous on the handle's stream: row k gets n_in[k] symbols."""
        n = self._counts(n_in)
        check(lib().sdr_eq_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), _ptr(d_err),
                                       out_stride), "sdr_eq_process_dev")

class Vit(_Handle):
    """Viterbi decoder bank (sdr_vit): soft-decision decoding of C streams of one rate-1/n convolutional code.
    K: constraint length (3..9); gens: n generators in the octal convention (the MSB taps the current input, e.g.
    (0o133, 0o171)); depth: the decision depth L (a multiple of 32, 32..512); scale: sigma, one or one per channel (soft
    values are quantised as rint(clamp(x sigma, -127, 127)), positive favouring bit 0); zero_start: the encoder starts
    in state 0 (else every state is equally likely).  A step is n f32 values; complex64 rows at n = 2 are one step per
    symbol (I -> c_0, Q -> c_1).  process returns the released bits, one uint8 (0 or 1) each; after T steps
    max(0, 32 floor(T/32) - L) bits are out, and finish releases the rest.  See include/sdr_b200.h."""

    _abi = "vit"

    def __init__(self, K, gens, depth, scale=1.0, n_channels=None, zero_start=True, device=0, stream=None):
        self._gens = np.ascontiguousarray(gens, np.uint32).ravel()
        self._scale = np.ascontiguousarray(np.atleast_1d(np.asarray(scale, np.float32)))
        self.K, self.n, self.depth = int(K), int(self._gens.size), int(depth)
        self.n_channels = int(n_channels) if n_channels is not None else int(self._scale.size)
        cfg = F.VitConfig(self.K, self._gens.ctypes.data, self._gens.size, self.depth, self._scale.ctypes.data,
                          self._scale.size, int(bool(zero_start)), self.n_channels, device, _stream_ptr(stream))
        self._create(cfg)

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def output_count(self, n_in):
        """bits the next call of n_in steps (an int, or C counts) releases per channel; no device work"""
        n = self._counts(n_in)
        out = np.empty(self.n_channels, np.uintp)
        check(lib().sdr_vit_output_count(self.h, n.ctypes.data, out.ctypes.data), "sdr_vit_output_count")
        return out.astype(np.int64)

    def process(self, rows):
        """rows: f32 [C, steps, n] or [C, steps * n], complex64 [C, steps] at n = 2, or a list of C such rows of any
        lengths -> a list of C uint8 arrays of released bits"""
        if isinstance(rows, np.ndarray) and self.n_channels == 1 and (rows.ndim == 1 or (
                rows.ndim == 2 and rows.shape[1] == self.n and rows.dtype != np.complex64)):
            rows = rows[None]
        rows = [np.ascontiguousarray(r).view(np.float32).ravel() if np.iscomplexobj(r)
                else np.ascontiguousarray(r, np.float32).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        if any(r.size % self.n for r in rows):
            raise ValueError("rows: whole steps of %d values expected" % self.n)
        n = np.array([r.size // self.n for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        x = np.zeros((self.n_channels, stride * self.n), np.float32)
        for k, r in enumerate(rows):
            x[k, :r.size] = r
        cnt = self.output_count(n)
        ostride = max(int(cnt.max()), 4)
        ostride += -ostride % 4
        y = np.empty((self.n_channels, ostride), np.uint8)
        got = np.empty(self.n_channels, np.uintp)
        check(lib().sdr_vit_process(self.h, x.ctypes.data, n.ctypes.data, stride, y.ctypes.data, ostride,
                                    got.ctypes.data), "sdr_vit_process")
        return [y[k, :int(got[k])].copy() for k in range(self.n_channels)]

    def process_dev(self, d_in, n_in, in_stride, d_out, out_stride):
        """device-resident: d_in C rows of in_stride steps (n f32 each), row k of n_in (an int, or C counts) steps;
        d_out C rows of out_stride bytes (a multiple of 4 when C > 1).  Asynchronous on the handle's stream; returns the
        C bit counts written, known on the host"""
        n = self._counts(n_in)
        got = np.empty(self.n_channels, np.uintp)
        check(lib().sdr_vit_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), out_stride,
                                        got.ctypes.data), "sdr_vit_process_dev")
        return got.astype(np.int64)

    def _which(self, which):
        return None if which is None else np.ascontiguousarray(np.broadcast_to(
            np.asarray(which, bool), (self.n_channels,)), np.uint8)

    def finish(self, which=None, terminated=True):
        """the remaining bits of the channels in `which` (C booleans; None: all), traced back from state 0
        (terminated) or from the best state; those channels return to their creation state.  A list of C uint8 arrays
        (empty for channels not listed)"""
        w = self._which(which)
        cap = self.depth + 32
        y = np.empty((self.n_channels, cap), np.uint8)
        got = np.empty(self.n_channels, np.uintp)
        check(lib().sdr_vit_finish(self.h, None if w is None else w.ctypes.data, int(bool(terminated)), y.ctypes.data,
                                   cap, got.ctypes.data), "sdr_vit_finish")
        return [y[k, :int(got[k])].copy() for k in range(self.n_channels)]

    def finish_dev(self, d_out, out_stride, which=None, terminated=True):
        """finish into device rows d_out (C rows of out_stride bytes, >= depth + 31); asynchronous; returns the C
        counts"""
        w = self._which(which)
        got = np.empty(self.n_channels, np.uintp)
        check(lib().sdr_vit_finish_dev(self.h, None if w is None else w.ctypes.data, int(bool(terminated)),
                                       _ptr(d_out), out_stride, got.ctypes.data), "sdr_vit_finish_dev")
        return got.astype(np.int64)


FSYNC_RECORD = np.dtype([("pos", "<u8"), ("out_index", "<u8"), ("corr", "<f4", (2,)), ("rho", "<f4"),
                         ("rot", "<u2"), ("kind", "<u2")])


class Fsync(_Handle):
    """Frame synchronizer bank (sdr_fsync): per channel, finds a known sync word by correlation, tracks frames with a
    search -> verify -> lock -> flywheel state machine and emits each frame's payload derotated by the rotation read
    from the correlation's phase.  words: Lp complex values (shared) or [C, Lp]; params: one
    (F, M, th_search, th_check, V, max_miss, W) or one per channel.  process returns the payload symbols and the
    decision records (FSYNC_RECORD: pos, out_index, corr, rho, rot, kind); see include/sdr_b200.h."""

    _abi = "fsync"
    SEARCH, VERIFY, LOCK = 0, 1, 2
    HIT, VERIFY_PASS, VERIFY_FAIL, LOCK_PASS, LOCK_MISS, LOCK_LOST = 1, 2, 3, 4, 5, 6

    def __init__(self, words, params, n_channels=None, device=0, stream=None):
        w = np.ascontiguousarray(words, np.complex64)
        w = w[None] if w.ndim == 1 else w
        prm = [params] if np.ndim(params[0]) == 0 else list(params)
        c = int(n_channels) if n_channels is not None else max(len(w), len(prm))
        self.n_channels, self.word_len = c, int(w.shape[1])
        self._words = w
        self._params = (F.FsyncParams * len(prm))(*[F.FsyncParams(int(p[0]), int(p[1]), float(p[2]), float(p[3]),
                                                                   int(p[4]), int(p[5]), int(p[6])) for p in prm])
        cfg = F.FsyncConfig(self.word_len, w.ctypes.data, len(w), C.addressof(self._params), len(prm), c, device,
                            _stream_ptr(stream))
        self._create(cfg)

    def _counts(self, n_in):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, np.int64), (self.n_channels,)), np.uintp)

    def max_output(self, n_in):
        """(payload bounds, record bounds): numpy arrays of C for the next n_in symbols (an int, or one per channel)"""
        n = self._counts(n_in)
        pc, rc = np.zeros(self.n_channels, np.uintp), np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fsync_max_output(self.h, n.ctypes.data, pc.ctypes.data, rc.ctypes.data),
              "sdr_fsync_max_output")
        return pc.astype(np.int64), rc.astype(np.int64)

    def state(self, k):
        """(state, v or m, sigma or e, R, symbols consumed, payload total) of channel k"""
        s = F.FsyncState()
        check(lib().sdr_fsync_get_state(self.h, int(k), C.byref(s)), "sdr_fsync_get_state")
        return s.state, s.count, s.pos, s.rot, s.consumed, s.payload

    def process(self, rows, records=True):
        """rows: complex64 [C, n] or a list of C rows of any lengths -> (payloads, records): lists of C complex64
        arrays and C FSYNC_RECORD arrays (None when records is False)"""
        if isinstance(rows, np.ndarray) and rows.ndim == 1 and self.n_channels == 1:
            rows = rows[None]
        rows = [np.ascontiguousarray(r, np.complex64).ravel() for r in rows]
        if len(rows) != self.n_channels:
            raise ValueError("rows: %d channels expected" % self.n_channels)
        n = np.array([r.size for r in rows], np.uintp)
        stride = max(int(n.max()), 1)
        x = np.zeros((self.n_channels, stride), np.complex64)
        for k, r in enumerate(rows):
            x[k, :r.size] = r
        pc, rc = self.max_output(n)
        cap, rcap = max(int(pc.max()), 1), max(int(rc.max()), 1)
        y = np.empty((self.n_channels, cap), np.complex64)
        rec = np.empty((self.n_channels, rcap), FSYNC_RECORD) if records else None
        got, rgot = np.zeros(self.n_channels, np.uintp), np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fsync_process(self.h, x.ctypes.data, n.ctypes.data, stride, y.ctypes.data, cap, cap,
                                      got.ctypes.data, None if rec is None else rec.ctypes.data, rcap, rcap,
                                      rgot.ctypes.data), "sdr_fsync_process")
        return ([y[k, :int(got[k])].copy() for k in range(self.n_channels)],
                None if rec is None else [rec[k, :int(rgot[k])].copy() for k in range(self.n_channels)])

    def process_dev(self, d_in, n_in, in_stride, d_out, out_cap, out_stride, d_rec=None, rec_cap=0, rec_stride=0):
        """device-resident: d_in C rows of in_stride complex64, row k of n_in (an int, or C counts) symbols; d_out C
        rows of out_stride complex64 (out_cap >= the payload bound); d_rec (C rows of rec_stride 32-byte records, e.g.
        a uint8 tensor [C, rec_stride, 32]) may be None.  Returns (payload counts, record counts), numpy arrays of C,
        once they are known, which synchronises the handle's stream."""
        n = self._counts(n_in)
        got, rgot = np.zeros(self.n_channels, np.uintp), np.zeros(self.n_channels, np.uintp)
        check(lib().sdr_fsync_process_dev(self.h, _ptr(d_in), n.ctypes.data, in_stride, _ptr(d_out), out_cap,
                                          out_stride, got.ctypes.data, _ptr(d_rec), rec_cap, rec_stride,
                                          rgot.ctypes.data), "sdr_fsync_process_dev")
        return got.astype(np.int64), rgot.astype(np.int64)


class FmStereo:
    """The FM broadcast stereo receiver of src/main.rs:32-81 for a batch of stations, device-resident end to end:
    u8 IQ -> Pll demodulator -> /75000 -> SincFastest to 144 kHz -> pilot Pll + (mono, diff) -> SincBest to 48 kHz ->
    Lr de-emphasis -> (left, right)."""

    def __init__(self, n_stations=1, rate=1.8e6, pilot=0.0, fast_math=True, device=0, stream=None):
        self.n_stations = int(n_stations)
        cfg = F.FmConfig(self.n_stations, rate, pilot, 0 if fast_math else F.PLL_F64_MATH, device, _stream_ptr(stream))
        err = C.c_int(0)
        self.h = lib().sdr_fm_create(C.byref(cfg), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_fm_create")

    @property
    def output_rate(self):
        return lib().sdr_fm_output_rate(self.h)

    def max_output(self, n):
        return lib().sdr_fm_max_output(self.h, n)

    def process(self, iq, end_of_input=False):
        """iq: uint8 [2n] or [n_stations, 2n] -> float32 [n_out, 2] or [n_stations, n_out, 2] (left, right) at 48 kHz"""
        iq = np.ascontiguousarray(iq, np.uint8)
        rows = iq.reshape(self.n_stations, -1)
        n = rows.shape[1] // 2
        cap = self.max_output(n)
        out = np.empty((self.n_stations, cap, 2), np.float32)
        got = C.c_size_t(0)
        check(lib().sdr_fm_process(self.h, rows.ctypes.data, n, rows.shape[1], out.ctypes.data, cap, cap,
                                   C.byref(got), int(bool(end_of_input))), "sdr_fm_process")
        out = out[:, :got.value]
        return out[0] if iq.ndim <= 1 else out

    def process_dev(self, d_iq, n, in_stride, d_out, out_cap, out_stride=None, end_of_input=False):
        got = C.c_size_t(0)
        check(lib().sdr_fm_process_dev(self.h, _ptr(d_iq), n, in_stride, _ptr(d_out), out_cap, out_stride or out_cap,
                                       C.byref(got), int(bool(end_of_input))), "sdr_fm_process_dev")
        return got.value

    def reset(self):
        check(lib().sdr_fm_reset(self.h), "sdr_fm_reset")

    def close(self):
        if getattr(self, "h", None):
            lib().sdr_fm_destroy(self.h)
            self.h = None

    __del__ = close


class Channelizer:
    """n_channels x (Fir<f32,Complex<f32>> -> Pll): BASELINE config 4."""

    def __init__(self, taps, design, n_channels, rate, input_format="c64", fast_math=True, strict=False,
                 device=0, stream=None):
        taps = np.ascontiguousarray(taps, np.float32)
        self._taps = taps
        self.n_channels = int(n_channels)
        self.fmt = _FMT_OF[input_format]
        fc = F.FirConfig(taps.ctypes.data, taps.size, 0, self.fmt, 1, self.n_channels,
                         F.FIR_STRICT_ORDER if strict else 0, device, _stream_ptr(stream))
        arr = (F.PllDesign * 1)(design._c())
        self._arr = arr
        pc = F.PllConfig(C.cast(arr, C.c_void_p), 1, self.n_channels, rate, 0 if fast_math else F.PLL_F64_MATH,
                         device, None)
        err = C.c_int(0)
        self.h = lib().sdr_channelizer_create(C.byref(fc), C.byref(pc), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_channelizer_create")

    def process(self, x):
        x = np.ascontiguousarray(x, _IN_DTYPE[self.fmt])
        per = 2 if self.fmt == F.FMT_U8IQ else 1
        rows = x.reshape(self.n_channels, -1)
        n = rows.shape[1] // per
        out = np.empty((self.n_channels, n), np.float32)
        locked = np.empty((self.n_channels, n), np.uint8)
        check(lib().sdr_channelizer_process(self.h, rows.ctypes.data, n, n, out.ctypes.data, locked.ctypes.data, n),
              "sdr_channelizer_process")
        return out, locked

    def process_dev(self, d_in, n, d_out, d_locked, in_stride=None, out_stride=None):
        check(lib().sdr_channelizer_process_dev(self.h, _ptr(d_in), n, in_stride or n, _ptr(d_out), _ptr(d_locked),
                                                out_stride or n), "sdr_channelizer_process_dev")

    def reset(self):
        check(lib().sdr_channelizer_reset(self.h), "sdr_channelizer_reset")

    def close(self):
        if getattr(self, "h", None):
            lib().sdr_channelizer_destroy(self.h)
            self.h = None

    __del__ = close


class ConverterType(enum.IntEnum):
    """resample::ConverterType (src/resample.rs:112-119)."""
    SincBestQuality = F.SRC_SINC_BEST_QUALITY
    SincMediumQuality = F.SRC_SINC_MEDIUM_QUALITY
    SincFastest = F.SRC_SINC_FASTEST
    ZeroOrderHold = F.SRC_ZERO_ORDER_HOLD
    Linear = F.SRC_LINEAR

    def name_str(self):
        return lib().sdr_src_get_name(int(self)).decode()

    def description(self):
        return lib().sdr_src_get_description(int(self)).decode()


class ResampleError(RuntimeError):
    def __init__(self, code):
        self.code = code
        msg = lib().sdr_src_strerror(code)
        super().__init__(msg.decode() if msg else "Unknown(%d)" % code)


class SampleRate(_Handle):
    """resample::SampleRate<A> (src/resample.rs:11-110).  channels: 1 for f32, 2 for Complex<f32>."""

    _abi = "src"

    def __init__(self, typ, channels, device=0, stream=None):
        self.channels = int(channels)
        err = C.c_int(0)
        self.h = lib().sdr_src_new_on(int(typ), self.channels, device, _stream_ptr(stream), C.byref(err))
        if not self.h:
            raise ResampleError(err.value)

    def process(self, ratio, inp, out_capacity):
        """SampleRate::process(ratio, &input, &mut output) (resample.rs:46-67): returns
        (input_frames_used, output[frames, channels]); end_of_input = input.is_empty()."""
        inp = np.ascontiguousarray(inp, np.float32).reshape(-1, self.channels)
        out = np.empty((max(out_capacity, 1), self.channels), np.float32)
        d = F.SrcData(inp.ctypes.data if inp.size else None, out.ctypes.data, inp.shape[0], out_capacity, 0, 0,
                      1 if inp.shape[0] == 0 else 0, ratio)
        rc = lib().sdr_src_process(self.h, C.byref(d))
        if rc != 0:
            raise ResampleError(rc)
        return d.input_frames_used, out[:d.output_frames_gen].copy()

    def process_dev(self, ratio, d_in, n_frames, d_out, out_capacity, end_of_input=False):
        """device-resident SampleRate::process: d_in / d_out are device buffers of interleaved f32 frames; the counts
        come back synchronously, the samples land asynchronously on the handle's stream.  Returns (used, generated)."""
        d = F.SrcData(_ptr(d_in) if n_frames else None, _ptr(d_out), int(n_frames), int(out_capacity), 0, 0,
                      1 if (end_of_input or n_frames == 0) else 0, ratio)
        rc = lib().sdr_src_process_dev(self.h, C.byref(d))
        if rc != 0:
            raise ResampleError(rc)
        return d.input_frames_used, d.output_frames_gen

    def reset(self):
        rc = lib().sdr_src_reset(self.h)
        if rc:
            raise ResampleError(rc)

    def try_clone(self):
        err = C.c_int(0)
        h = lib().sdr_src_clone(self.h, C.byref(err))
        if not h:
            raise ResampleError(err.value)
        return self._adopt(h)

    def set_ratio(self, ratio):
        rc = lib().sdr_src_set_ratio(self.h, ratio)
        if rc:
            raise ResampleError(rc)

    def get_channels(self):
        return lib().sdr_src_get_channels(self.h)

    def history_frames(self):
        return lib().sdr_src_history_frames(self.h)

    def set_exact(self, exact=True):
        """True: always the f64 kernels (the converter's specification up to the final f32 rounding); False (default):
        long integer-step calls on c64 data may take the tensor-core polyphase path (within 1e-5 of max|y|)"""
        rc = lib().sdr_src_set_exact(self.h, 1 if exact else 0)
        if rc:
            raise ResampleError(rc)

    def close(self):
        if self.h:
            lib().sdr_src_delete(self.h)
            self.h = None


def sinc_table(typ):
    tab = C.c_void_p()
    inc = C.c_int()
    n = lib().sdr_src_sinc_table(int(typ), C.byref(tab), C.byref(inc))
    arr = np.ctypeslib.as_array(C.cast(tab, C.POINTER(C.c_float)), shape=(n + 2,)).copy()
    return arr, inc.value, n


class Timer:
    """CUDA-event timer on a given stream (the stream kernels are launched on)."""

    def __init__(self, device=0, stream=None):
        err = C.c_int(0)
        self.h = lib().sdr_timer_create(device, _stream_ptr(stream), C.byref(err))
        if not self.h:
            raise SdrError(err.value, "sdr_timer_create")

    def begin(self):
        check(lib().sdr_timer_begin(self.h), "sdr_timer_begin")

    def end(self):
        ms = C.c_float(0)
        check(lib().sdr_timer_end(self.h, C.byref(ms)), "sdr_timer_end")
        return ms.value

    def close(self):
        if getattr(self, "h", None):
            lib().sdr_timer_destroy(self.h)
            self.h = None

    __del__ = close

//! gpu.rs -- safe wrappers a maintainer would add to the crate (`mod gpu;` in src/lib.rs).
//! NOT COMPILED HERE (no Rust toolchain in this image); kept deliberately thin so that everything with
//! behaviour lives behind the C ABI, where it is tested from C++ and Python.
//!
//! What changes in the reference tree:
//!   * src/resample.rs:1      `use libsamplerate_sys::*;`  ->  `use crate::sdr_b200_sys::{sdr_src_new as src_new,
//!                             sdr_src_process as src_process, sdr_src_reset as src_reset, sdr_src_clone as src_clone,
//!                             sdr_src_delete as src_delete, sdr_src_set_ratio as src_set_ratio,
//!                             sdr_src_get_channels as src_get_channels, sdr_src_strerror as src_strerror,
//!                             sdr_src_get_name as src_get_name, sdr_src_get_description as src_get_description,
//!                             sdr_src_get_version as src_get_version, SDR_SRC_STATE as SRC_STATE, SDR_SRC_DATA as SRC_DATA};`
//!                             (+ the five SRC_* converter constants).  Nothing else in resample.rs changes.
//!   * src/fft.rs:10-12       the rustfft planner + process become `gpu::fft_shifted(&data, rate)`.
//!   * src/signal/adapters/mod.rs  `Filter<S, Fir<..>>` gets a block-buffered `next()` (below), shaped exactly like
//!                             signal::Resample::next (src/signal/adapters/resample.rs:38-82).
use crate::sdr_b200_sys::*;
use crate::Signal;
use num::Complex;
use std::os::raw::c_void;

#[derive(Debug)]
pub struct Error(pub i32);
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter) -> std::fmt::Result {
        let s = unsafe { std::ffi::CStr::from_ptr(sdr_strerror(self.0)) };
        write!(f, "{}", s.to_string_lossy())
    }
}
fn check(rc: i32) -> Result<(), Error> { if rc == SDR_OK { Ok(()) } else { Err(Error(rc)) } }

/// sealed: sample / coefficient types the GPU path accepts (there is no CPU fallback)
pub trait GpuSample: Copy { const FMT: i32; }
impl GpuSample for f32 { const FMT: i32 = SDR_FMT_F32; }
impl GpuSample for Complex<f32> { const FMT: i32 = SDR_FMT_C64; }
pub trait GpuCoef: Copy { const COMPLEX: i32; }
impl GpuCoef for f32 { const COMPLEX: i32 = 0; }
impl GpuCoef for Complex<f32> { const COMPLEX: i32 = 1; }

/// filter::Fir<C, A> backed by the GPU: same constructor, plus a block `process` mirroring
/// resample::SampleRate::process (src/resample.rs:46-67).
pub struct GpuFir<C: GpuCoef, A: GpuSample> {
    h: *mut sdr_fir_t,
    _m: std::marker::PhantomData<(C, fn(A) -> A)>,
}
unsafe impl<C: GpuCoef, A: GpuSample> Send for GpuFir<C, A> {}

impl<C: GpuCoef, A: GpuSample> GpuFir<C, A> {
    pub fn new(coef: Vec<C>) -> Result<Self, Error> { Self::with_decimation(coef, 1, false) }
    pub fn with_decimation(coef: Vec<C>, wait: usize, input_u8iq: bool) -> Result<Self, Error> {
        let cfg = sdr_fir_config_t {
            taps: coef.as_ptr() as *const f32, n_taps: coef.len(), taps_complex: C::COMPLEX,
            input_format: if input_u8iq { SDR_FMT_U8IQ } else { A::FMT },
            decimation: wait, n_channels: 1, flags: 0, device: 0, stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_fir_create(&cfg, &mut err) };
        if h.is_null() { Err(Error(err)) } else { Ok(GpuFir { h, _m: std::marker::PhantomData }) }
    }
    /// output gets one element per kept input; returns inputs consumed
    pub fn process(&mut self, input: &[A], output: &mut Vec<A>) -> Result<usize, Error> {
        let n_out = unsafe { sdr_fir_output_count(self.h, input.len()) };
        output.clear();
        output.reserve(n_out);
        let (mut used, mut got) = (0usize, 0usize);
        check(unsafe {
            sdr_fir_process(self.h, input.as_ptr() as *const c_void, input.len(), input.len(),
                            output.as_mut_ptr() as *mut c_void, n_out, n_out, &mut used, &mut got)
        })?;
        unsafe { output.set_len(got) };
        Ok(used)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_fir_reset(self.h) }) }
}
impl<C: GpuCoef, A: GpuSample> Clone for GpuFir<C, A> {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_fir_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_fir_clone failed: {}", Error(err));
        GpuFir { h, _m: std::marker::PhantomData }
    }
}
impl<C: GpuCoef, A: GpuSample> Drop for GpuFir<C, A> {
    fn drop(&mut self) { unsafe { sdr_fir_destroy(self.h) } }
}

/// Block-buffered signal::Filter for a GPU FIR: pulls `block` samples upstream, one launch, serves one by one.
/// Same shape as signal::Resample::next (src/signal/adapters/resample.rs:38-82).
pub struct GpuFilter<S: Signal, C: GpuCoef> where S::Sample: GpuSample {
    signal: S,
    fir: GpuFir<C, S::Sample>,
    block: usize,
    input: Vec<S::Sample>,
    output: Vec<S::Sample>,
    next: usize,
}
impl<S: Signal, C: GpuCoef> Signal for GpuFilter<S, C> where S::Sample: GpuSample {
    type Sample = S::Sample;
    fn next(&mut self) -> Option<Self::Sample> {
        while self.next >= self.output.len() {
            self.input.clear();
            while self.input.len() < self.block {
                match self.signal.next() { Some(v) => self.input.push(v), None => break }
            }
            if self.input.is_empty() { return None; }
            self.fir.process(&self.input, &mut self.output).unwrap();
            self.next = 0;
        }
        let v = self.output[self.next];
        self.next += 1;
        Some(v)
    }
    fn rate(&self) -> f32 { self.signal.rate() }
}

/// Polyphase filter bank: channel k is Fir<Complex<f32>, Complex<f32>> with taps h[n] e^{+2 pi i k n / M} followed by
/// Decimate(wait), for k = 0..M-1, in one pass over the input.  `process` returns frames of M channels (or M rows of
/// frames with SDR_PFB_CHANNEL_MAJOR); blocks of any size give the same samples as one call.
pub struct GpuPfb {
    h: *mut sdr_pfb_t,
    m: usize,
    channel_major: bool,
}
unsafe impl Send for GpuPfb {}

impl GpuPfb {
    pub fn new(prototype: &[f32], channels: usize, wait: usize, input_u8iq: bool, flags: u32) -> Result<Self, Error> {
        let cfg = sdr_pfb_config_t {
            taps: prototype.as_ptr(), n_taps: prototype.len(), n_channels: channels, decimation: wait,
            input_format: if input_u8iq { SDR_FMT_U8IQ } else { SDR_FMT_C64 }, flags, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_pfb_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuPfb { h, m: channels, channel_major: flags & SDR_PFB_CHANNEL_MAJOR != 0 })
    }
    /// input: n samples (Complex<f32>, or 2n rtl_tcp bytes); output: replaced by frames x M (or M x frames)
    pub fn process<T: Copy>(&mut self, input: &[T], n: usize, output: &mut Vec<Complex<f32>>) -> Result<usize, Error> {
        let nf = unsafe { sdr_pfb_output_count(self.h, n) };
        output.clear();
        output.reserve(nf.max(1) * self.m);
        let mut got = 0usize;
        let stride = if self.channel_major { nf } else { self.m };
        check(unsafe {
            sdr_pfb_process(self.h, input.as_ptr() as *const c_void, n, output.as_mut_ptr() as *mut f32, nf, stride,
                            &mut got)
        })?;
        unsafe { output.set_len(got * self.m) };
        Ok(got)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_pfb_reset(self.h) }) }
}
impl Clone for GpuPfb {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_pfb_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_pfb_clone failed: {}", Error(err));
        GpuPfb { h, m: self.m, channel_major: self.channel_major }
    }
}
impl Drop for GpuPfb {
    fn drop(&mut self) { unsafe { sdr_pfb_destroy(self.h) } }
}

/// Polyphase synthesis bank, the inverse of GpuPfb: channel k is zero-stuffed by `interpolation` (D), filtered by
/// Fir<Complex<f32>, Complex<f32>> with taps f[n] e^{+2 pi i k n / M} and summed over k.  `process` takes frames of M
/// channels (or M rows of frames with SDR_PFS_CHANNEL_MAJOR) and returns D samples per frame; calls of any number of
/// frames give the same samples as one call.
pub struct GpuPfs {
    h: *mut sdr_pfs_t,
    m: usize,
    channel_major: bool,
}
unsafe impl Send for GpuPfs {}

impl GpuPfs {
    pub fn new(prototype: &[f32], channels: usize, interpolation: usize, flags: u32) -> Result<Self, Error> {
        let cfg = sdr_pfs_config_t {
            taps: prototype.as_ptr(), n_taps: prototype.len(), n_channels: channels, interpolation, flags, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_pfs_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuPfs { h, m: channels, channel_major: flags & SDR_PFS_CHANNEL_MAJOR != 0 })
    }
    /// input: n_frames frames of M (or M rows of n_frames); output: replaced by n_frames * D samples
    pub fn process(&mut self, input: &[Complex<f32>], n_frames: usize, output: &mut Vec<Complex<f32>>)
                   -> Result<usize, Error> {
        assert!(input.len() >= n_frames * self.m);
        let n = unsafe { sdr_pfs_output_count(self.h, n_frames) };
        output.clear();
        output.reserve(n.max(1));
        let mut got = 0usize;
        let stride = if self.channel_major { n_frames } else { self.m };
        check(unsafe {
            sdr_pfs_process(self.h, input.as_ptr() as *const f32, n_frames, stride, output.as_mut_ptr() as *mut f32, n,
                            &mut got)
        })?;
        unsafe { output.set_len(got) };
        Ok(got)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_pfs_reset(self.h) }) }
}
impl Clone for GpuPfs {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_pfs_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_pfs_clone failed: {}", Error(err));
        GpuPfs { h, m: self.m, channel_major: self.channel_major }
    }
}
impl Drop for GpuPfs {
    fn drop(&mut self) { unsafe { sdr_pfs_destroy(self.h) } }
}

/// Down-converter bank: channel k is the stream mixed down by a 64-bit NCO at freqs[k] (what a caller writes with
/// Signal::map over an oscillator), Fir<Complex<f32>, f32>(h_k) and Decimate(wait), for all channels in one pass over
/// the input.  taps: one row of n_taps (shared) or one row per channel.  `process` returns channels rows of outputs
/// (channel-major); blocks of any size give the same samples as one call.
pub struct GpuDdc {
    h: *mut sdr_ddc_t,
    c: usize,
}
unsafe impl Send for GpuDdc {}

impl GpuDdc {
    pub fn new(taps: &[f32], n_taps: usize, freqs: &[f64], rate: f64, wait: usize, input_u8iq: bool,
               first_sample: u64, flags: u32) -> Result<Self, Error> {
        let inc: Vec<u64> = freqs.iter().map(|&f| unsafe { sdr_ddc_phase_increment(f, rate) }).collect();
        let cfg = sdr_ddc_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: if n_taps == 0 { 0 } else { taps.len() / n_taps },
            phase_inc: inc.as_ptr(), n_channels: freqs.len(), decimation: wait, first_sample,
            input_format: if input_u8iq { SDR_FMT_U8IQ } else { SDR_FMT_C64 }, flags, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_ddc_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuDdc { h, c: freqs.len() })
    }
    /// input: n samples (Complex<f32>, or 2n rtl_tcp bytes); output: replaced by channels x outputs
    pub fn process<T: Copy>(&mut self, input: &[T], n: usize, output: &mut Vec<Complex<f32>>) -> Result<usize, Error> {
        let nf = unsafe { sdr_ddc_output_count(self.h, n) };
        output.clear();
        output.reserve(nf.max(1) * self.c);
        let mut got = 0usize;
        check(unsafe {
            sdr_ddc_process(self.h, input.as_ptr() as *const c_void, n, output.as_mut_ptr() as *mut f32, nf, nf.max(1),
                            &mut got)
        })?;
        unsafe { output.set_len(got * self.c) };
        Ok(got)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_ddc_reset(self.h) }) }
}
impl Clone for GpuDdc {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_ddc_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_ddc_clone failed: {}", Error(err));
        GpuDdc { h, c: self.c }
    }
}
impl Drop for GpuDdc {
    fn drop(&mut self) { unsafe { sdr_ddc_destroy(self.h) } }
}

/// Up-converter bank, the transpose of GpuDdc: channel k is zero-stuffed by `interpolation` (I; sample m at index
/// (m+1) I - 1), filtered by Fir<f32, Complex<f32>>(h_k), mixed up by a 64-bit NCO at freqs[k] and the channels are
/// summed into one stream.  taps: one row of n_taps (shared) or one row per channel.  `process` takes channels rows of
/// frames (the rows GpuDdc returns) and returns I samples per frame; calls of any number of frames give the same
/// samples as one call.  first_sample: absolute index of the first output (after GpuDdc, its first_sample minus the
/// filter cascade's delay).
pub struct GpuDuc {
    h: *mut sdr_duc_t,
    c: usize,
}
unsafe impl Send for GpuDuc {}

impl GpuDuc {
    pub fn new(taps: &[f32], n_taps: usize, freqs: &[f64], rate: f64, interpolation: usize, first_sample: u64)
               -> Result<Self, Error> {
        let inc: Vec<u64> = freqs.iter().map(|&f| unsafe { sdr_ddc_phase_increment(f, rate) }).collect();
        let cfg = sdr_duc_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: if n_taps == 0 { 0 } else { taps.len() / n_taps },
            phase_inc: inc.as_ptr(), n_channels: freqs.len(), interpolation, first_sample, flags: 0, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_duc_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuDuc { h, c: freqs.len() })
    }
    /// input: channels rows of n_frames, row stride `stride` (>= n_frames); output: replaced by n_frames * I samples
    pub fn process(&mut self, input: &[Complex<f32>], n_frames: usize, stride: usize, output: &mut Vec<Complex<f32>>)
                   -> Result<usize, Error> {
        assert!(n_frames == 0 || input.len() >= (self.c - 1) * stride + n_frames);
        let n = unsafe { sdr_duc_output_count(self.h, n_frames) };
        output.clear();
        output.reserve(n.max(1));
        let mut got = 0usize;
        check(unsafe {
            sdr_duc_process(self.h, input.as_ptr() as *const f32, n_frames, stride, output.as_mut_ptr() as *mut f32, n,
                            &mut got)
        })?;
        unsafe { output.set_len(got) };
        Ok(got)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_duc_reset(self.h) }) }
}
impl Clone for GpuDuc {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_duc_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_duc_clone failed: {}", Error(err));
        GpuDuc { h, c: self.c }
    }
}
impl Drop for GpuDuc {
    fn drop(&mut self) { unsafe { sdr_duc_destroy(self.h) } }
}

/// window(n) -> decimate(hop) -> map(fft::fft) -> |.|^2 -> mean of `average` behind sdr_psd_*: averaged power spectra
/// of n f32 bins (shifted and 1/n-scaled like fft::fft's 1/sqrt(n) with SDR_PSD_SHIFT | SDR_PSD_NORM).  taper: n real
/// values or empty (rectangular).  `process` appends the spectra the block completes; blocks of any size give the same
/// bits as one call.
pub struct GpuPsd {
    h: *mut sdr_psd_t,
    n: usize,
}
unsafe impl Send for GpuPsd {}

impl GpuPsd {
    pub fn new(n: usize, hop: usize, average: usize, taper: &[f32], input_u8iq: bool, flags: u32) -> Result<Self, Error> {
        if !taper.is_empty() && taper.len() != n { return Err(Error(100)); }  // SDR_ERR_INVALID_ARG: the C side copies n values
        let cfg = sdr_psd_config_t {
            n, hop, average, window: if taper.is_empty() { std::ptr::null() } else { taper.as_ptr() },
            input_format: if input_u8iq { SDR_FMT_U8IQ } else { SDR_FMT_C64 }, flags, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_psd_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuPsd { h, n })
    }
    /// input: m samples (Complex<f32>, or 2m rtl_tcp bytes); the spectra are appended to output
    pub fn process<T: Copy>(&mut self, input: &[T], m: usize, output: &mut Vec<f32>) -> Result<usize, Error> {
        let ns = unsafe { sdr_psd_output_count(self.h, m) };
        let at = output.len();
        output.resize(at + ns.max(1) * self.n, 0.0);
        let mut got = 0usize;
        check(unsafe {
            sdr_psd_process(self.h, input.as_ptr() as *const c_void, m, output[at..].as_mut_ptr(), ns, self.n, &mut got)
        })?;
        output.truncate(at + got * self.n);
        Ok(got)
    }
    pub fn last_path(&self) -> i32 { unsafe { sdr_psd_last_path(self.h) } }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_psd_reset(self.h) }) }
}
impl Clone for GpuPsd {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_psd_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_psd_clone failed: {}", Error(err));
        GpuPsd { h, n: self.n }
    }
}
impl Drop for GpuPsd {
    fn drop(&mut self) { unsafe { sdr_psd_destroy(self.h) } }
}

/// Fast-convolution channel bank: GpuDdc's channels with one decimation per channel, by overlap-save.  Outputs are
/// released per block of P inputs (sdr_fcfb_geometry); feed N zeros to drain a finite stream.
pub struct GpuFcfb {
    h: *mut sdr_fcfb_t,
    c: usize,
}
unsafe impl Send for GpuFcfb {}

impl GpuFcfb {
    /// taps: one row of n_taps (shared) or one row per channel; freqs in Hz at `rate`; one decimation per channel
    pub fn new(taps: &[f32], n_taps: usize, freqs: &[f64], rate: f64, decimation: &[usize], input_u8iq: bool,
               first_sample: u64) -> Result<Self, Error> {
        if decimation.len() != freqs.len() || n_taps == 0 { return Err(Error(100)); }
        let inc: Vec<u64> = freqs.iter().map(|&f| unsafe { sdr_ddc_phase_increment(f, rate) }).collect();
        let cfg = sdr_fcfb_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: taps.len() / n_taps, phase_inc: inc.as_ptr(),
            decimation: decimation.as_ptr(), n_channels: freqs.len(), first_sample,
            input_format: if input_u8iq { SDR_FMT_U8IQ } else { SDR_FMT_C64 }, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_fcfb_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuFcfb { h, c: freqs.len() })
    }
    /// input: m samples (Complex<f32>, or 2m rtl_tcp bytes); channel k's released outputs are appended to output[k]
    pub fn process<T: Copy>(&mut self, input: &[T], m: usize, output: &mut [Vec<Complex<f32>>]) -> Result<(), Error> {
        let mut cnt = vec![0usize; self.c];
        check(unsafe { sdr_fcfb_output_count(self.h, m, cnt.as_mut_ptr()) })?;
        let cap = cnt.iter().copied().max().unwrap_or(0).max(1);
        let mut rows = vec![Complex::new(0.0f32, 0.0); cap * self.c];
        let mut got = vec![0usize; self.c];
        check(unsafe {
            sdr_fcfb_process(self.h, input.as_ptr() as *const c_void, m, rows.as_mut_ptr() as *mut f32, cap, cap,
                             got.as_mut_ptr())
        })?;
        for (k, out) in output.iter_mut().enumerate().take(self.c) {
            out.extend_from_slice(&rows[k * cap..k * cap + got[k]]);
        }
        Ok(())
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_fcfb_reset(self.h) }) }
}
impl Clone for GpuFcfb {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_fcfb_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_fcfb_clone failed: {}", Error(err));
        GpuFcfb { h, c: self.c }
    }
}
impl Drop for GpuFcfb {
    fn drop(&mut self) { unsafe { sdr_fcfb_destroy(self.h) } }
}

/// Fast-convolution synthesis bank, the inverse of GpuFcfb: GpuDuc's channels with one interpolation per channel, by
/// overlap-save.  A call advances by n_time output positions (a multiple of lcm(I_k); row k holds n_time / I_k frames,
/// the rows GpuFcfb returns) and appends the outputs of the blocks it completes; feed zero frames covering N positions
/// to drain a finite stream.  first_sample: absolute index of the first output (after GpuFcfb, its first_sample minus
/// the filter cascade's delay).
pub struct GpuFcsb {
    h: *mut sdr_fcsb_t,
    i: Vec<usize>,
}
unsafe impl Send for GpuFcsb {}

impl GpuFcsb {
    /// taps: one row of n_taps (shared) or one row per channel; freqs in Hz at `rate`; one interpolation per channel
    pub fn new(taps: &[f32], n_taps: usize, freqs: &[f64], rate: f64, interpolation: &[usize], first_sample: u64)
               -> Result<Self, Error> {
        if interpolation.len() != freqs.len() || n_taps == 0 { return Err(Error(100)); }
        let inc: Vec<u64> = freqs.iter().map(|&f| unsafe { sdr_ddc_phase_increment(f, rate) }).collect();
        let cfg = sdr_fcsb_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: taps.len() / n_taps, phase_inc: inc.as_ptr(),
            interpolation: interpolation.as_ptr(), n_channels: freqs.len(), first_sample, device: 0,
            stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_fcsb_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuFcsb { h, i: interpolation.to_vec() })
    }
    /// input: one row per channel, row k n_time / I_k frames at row stride `stride` (>= the longest row); the
    /// released outputs are appended to output
    pub fn process(&mut self, input: &[Complex<f32>], n_time: usize, stride: usize, output: &mut Vec<Complex<f32>>)
                   -> Result<usize, Error> {
        let last = self.i.len() - 1;
        assert!(n_time == 0 || input.len() >= last * stride + n_time / self.i[last]);
        let n = unsafe { sdr_fcsb_output_count(self.h, n_time) };
        let at = output.len();
        output.resize(at + n.max(1), Complex::new(0.0, 0.0));
        let mut got = 0usize;
        check(unsafe {
            sdr_fcsb_process(self.h, input.as_ptr() as *const f32, n_time, stride, output[at..].as_mut_ptr() as *mut f32,
                             n, &mut got)
        })?;
        output.truncate(at + got);
        Ok(got)
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_fcsb_reset(self.h) }) }
}
impl Clone for GpuFcsb {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_fcsb_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_fcsb_clone failed: {}", Error(err));
        GpuFcsb { h, i: self.i.clone() }
    }
}
impl Drop for GpuFcsb {
    fn drop(&mut self) { unsafe { sdr_fcsb_destroy(self.h) } }
}

/// Rational resampler bank: channel k zero-stuffed by I_k, filtered by its real taps and decimated by D_k (upfirdn).
/// After n frames a channel has released floor(n I_k / D_k) outputs; the taps carry the gain I_k.
pub struct GpuRrb {
    h: *mut sdr_rrb_t,
    c: usize,
}
unsafe impl Send for GpuRrb {}

impl GpuRrb {
    /// taps: one row of n_taps (shared) or one row per channel; one interpolation and one decimation per channel
    pub fn new(taps: &[f32], n_taps: usize, interpolation: &[usize], decimation: &[usize]) -> Result<Self, Error> {
        if interpolation.len() != decimation.len() || n_taps == 0 { return Err(Error(100)); }
        let cfg = sdr_rrb_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: taps.len() / n_taps, interpolation: interpolation.as_ptr(),
            decimation: decimation.as_ptr(), n_channels: interpolation.len(), device: 0, stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_rrb_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuRrb { h, c: interpolation.len() })
    }
    /// input: one row per channel, row k of n_in[k] frames at row stride `stride` (>= the longest row); channel k's
    /// outputs are appended to output[k]
    pub fn process(&mut self, input: &[Complex<f32>], n_in: &[usize], stride: usize,
                   output: &mut [Vec<Complex<f32>>]) -> Result<(), Error> {
        assert!(n_in.len() == self.c);
        assert!(n_in.iter().enumerate().all(|(k, &n)| n == 0 || input.len() >= k * stride + n));
        let mut cnt = vec![0usize; self.c];
        check(unsafe { sdr_rrb_output_count(self.h, n_in.as_ptr(), cnt.as_mut_ptr()) })?;
        let cap = cnt.iter().copied().max().unwrap_or(0).max(1);
        let mut rows = vec![Complex::new(0.0f32, 0.0); cap * self.c];
        let mut got = vec![0usize; self.c];
        check(unsafe {
            sdr_rrb_process(self.h, input.as_ptr() as *const f32, n_in.as_ptr(), stride, rows.as_mut_ptr() as *mut f32,
                            cap, cap, got.as_mut_ptr())
        })?;
        for (k, out) in output.iter_mut().enumerate().take(self.c) {
            out.extend_from_slice(&rows[k * cap..k * cap + got[k]]);
        }
        Ok(())
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_rrb_reset(self.h) }) }
}
impl Clone for GpuRrb {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_rrb_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_rrb_clone failed: {}", Error(err));
        GpuRrb { h, c: self.c }
    }
}
impl Drop for GpuRrb {
    fn drop(&mut self) { unsafe { sdr_rrb_destroy(self.h) } }
}

/// Arbitrary-ratio resampler bank: channel k resampled by its own step (input frames per output, exact in units of
/// 2^-64) with real taps designed at `phases` times the input rate, interpolated between adjacent phases.  After n
/// frames a channel has released #{r : tau(r) < n} outputs; unit gain needs taps summing to `phases`.
pub struct GpuArb {
    h: *mut sdr_arb_t,
    c: usize,
}
unsafe impl Send for GpuArb {}

impl GpuArb {
    /// rate_in / rate_out to the nearest 2^-64
    pub fn step(rate_in: f64, rate_out: f64) -> Result<sdr_arb_time_t, Error> {
        let mut t = sdr_arb_time_t::default();
        check(unsafe { sdr_arb_step(rate_in, rate_out, &mut t) })?;
        Ok(t)
    }
    /// taps: one row of n_taps (shared) or one row per channel; one step per channel; first: empty (all 0) or one
    /// position per channel
    pub fn new(taps: &[f32], n_taps: usize, phases: usize, steps: &[sdr_arb_time_t], first: &[sdr_arb_time_t])
               -> Result<Self, Error> {
        if n_taps == 0 || (!first.is_empty() && first.len() != steps.len()) { return Err(Error(100)); }
        let cfg = sdr_arb_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: taps.len() / n_taps, phases, step: steps.as_ptr(),
            first: if first.is_empty() { std::ptr::null() } else { first.as_ptr() }, n_channels: steps.len(),
            device: 0, stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_arb_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuArb { h, c: steps.len() })
    }
    /// new steps from each channel's next unreleased output on
    pub fn set_steps(&mut self, steps: &[sdr_arb_time_t]) -> Result<(), Error> {
        assert!(steps.len() == self.c);
        check(unsafe { sdr_arb_set_steps(self.h, steps.as_ptr()) })
    }
    /// input: one row per channel, row k of n_in[k] frames at row stride `stride` (>= the longest row); channel k's
    /// outputs are appended to output[k]
    pub fn process(&mut self, input: &[Complex<f32>], n_in: &[usize], stride: usize,
                   output: &mut [Vec<Complex<f32>>]) -> Result<(), Error> {
        assert!(n_in.len() == self.c);
        assert!(n_in.iter().enumerate().all(|(k, &n)| n == 0 || input.len() >= k * stride + n));
        let mut cnt = vec![0usize; self.c];
        check(unsafe { sdr_arb_output_count(self.h, n_in.as_ptr(), cnt.as_mut_ptr()) })?;
        let cap = cnt.iter().copied().max().unwrap_or(0).max(1);
        let mut rows = vec![Complex::new(0.0f32, 0.0); cap * self.c];
        let mut got = vec![0usize; self.c];
        check(unsafe {
            sdr_arb_process(self.h, input.as_ptr() as *const f32, n_in.as_ptr(), stride, rows.as_mut_ptr() as *mut f32,
                            cap, cap, got.as_mut_ptr())
        })?;
        for (k, out) in output.iter_mut().enumerate().take(self.c) {
            out.extend_from_slice(&rows[k * cap..k * cap + got[k]]);
        }
        Ok(())
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_arb_reset(self.h) }) }
}
impl Clone for GpuArb {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_arb_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_arb_clone failed: {}", Error(err));
        GpuArb { h, c: self.c }
    }
}
impl Drop for GpuArb {
    fn drop(&mut self) { unsafe { sdr_arb_destroy(self.h) } }
}

/// Symbol timing recovery bank: a Gardner loop per channel steering `GpuArb`'s interpolator on the exact 64.64 time
/// base.  Channel k: matched-filter taps at `phases` times the input rate, a nominal period (`GpuArb::step(rate,
/// symbol_rate)`), a first position and loop parameters; each call appends the released symbols, their exact positions
/// and the detector outputs.  Counts come from the device, so every call synchronises.
pub struct GpuTsync {
    h: *mut sdr_tsync_t,
    c: usize,
}
unsafe impl Send for GpuTsync {}

impl GpuTsync {
    /// (kp, ki) of the second-order loop for noise bandwidth bn_t, damping zeta and detector slope ted_gain
    pub fn loop_design(bn_t: f64, zeta: f64, ted_gain: f64, period_frames: f64) -> Result<(f32, f32), Error> {
        let (mut kp, mut ki) = (0.0f32, 0.0f32);
        check(unsafe { sdr_tsync_loop_design(bn_t, zeta, ted_gain, period_frames, &mut kp, &mut ki) })?;
        Ok((kp, ki))
    }
    /// taps: one row of n_taps (shared) or one row per channel; one period per channel; loops: one (shared) or one per
    /// channel; first: empty (all 0) or one position per channel
    pub fn new(taps: &[f32], n_taps: usize, phases: usize, periods: &[sdr_arb_time_t], loops: &[sdr_tsync_loop_t],
               first: &[sdr_arb_time_t]) -> Result<Self, Error> {
        if n_taps == 0 || (!first.is_empty() && first.len() != periods.len()) { return Err(Error(100)); }
        let cfg = sdr_tsync_config_t {
            taps: taps.as_ptr(), n_taps, n_tap_sets: taps.len() / n_taps, phases, period: periods.as_ptr(),
            first: if first.is_empty() { std::ptr::null() } else { first.as_ptr() }, loops: loops.as_ptr(),
            n_loops: loops.len(), n_channels: periods.len(), device: 0, stream: std::ptr::null_mut(),
        };
        let mut err = 0;
        let h = unsafe { sdr_tsync_create(&cfg, &mut err) };
        if h.is_null() { return Err(Error(err)); }
        Ok(GpuTsync { h, c: periods.len() })
    }
    /// next unreleased position and period offset v (units of 2^-40 frames) of one channel
    pub fn state(&mut self, k: usize) -> Result<(sdr_arb_time_t, i64), Error> {
        let mut t = sdr_arb_time_t::default();
        let mut v = 0i64;
        check(unsafe { sdr_tsync_get_state(self.h, k, &mut t, &mut v) })?;
        Ok((t, v))
    }
    /// input: one row per channel, row k of n_in[k] frames at row stride `stride` (>= the longest row); channel k's
    /// symbols, positions and errors are appended to sym[k], pos[k] and err[k]
    pub fn process(&mut self, input: &[Complex<f32>], n_in: &[usize], stride: usize, sym: &mut [Vec<Complex<f32>>],
                   pos: &mut [Vec<sdr_arb_time_t>], err: &mut [Vec<f32>]) -> Result<(), Error> {
        assert!(n_in.len() == self.c);
        assert!(n_in.iter().enumerate().all(|(k, &n)| n == 0 || input.len() >= k * stride + n));
        let mut caps = vec![0usize; self.c];
        check(unsafe { sdr_tsync_max_output(self.h, n_in.as_ptr(), caps.as_mut_ptr()) })?;
        let cap = caps.iter().copied().max().unwrap_or(0).max(1);
        let mut s = vec![Complex::new(0.0f32, 0.0); cap * self.c];
        let mut p = vec![sdr_arb_time_t::default(); cap * self.c];
        let mut e = vec![0.0f32; cap * self.c];
        let mut got = vec![0usize; self.c];
        check(unsafe {
            sdr_tsync_process(self.h, input.as_ptr() as *const f32, n_in.as_ptr(), stride, s.as_mut_ptr() as *mut f32,
                              p.as_mut_ptr(), e.as_mut_ptr(), cap, cap, got.as_mut_ptr())
        })?;
        for k in 0..self.c {
            let r = k * cap..k * cap + got[k];
            sym[k].extend_from_slice(&s[r.clone()]);
            pos[k].extend_from_slice(&p[r.clone()]);
            err[k].extend_from_slice(&e[r]);
        }
        Ok(())
    }
    pub fn reset(&mut self) -> Result<(), Error> { check(unsafe { sdr_tsync_reset(self.h) }) }
}
impl Clone for GpuTsync {
    fn clone(&self) -> Self {
        let mut err = 0;
        let h = unsafe { sdr_tsync_clone(self.h, &mut err) };
        assert!(!h.is_null(), "sdr_tsync_clone failed: {}", Error(err));
        GpuTsync { h, c: self.c }
    }
}
impl Drop for GpuTsync {
    fn drop(&mut self) { unsafe { sdr_tsync_destroy(self.h) } }
}

/// body of fft::fft after `let mut data: Vec<_> = input.iter().collect();` (src/fft.rs:8-27)
pub fn fft_shifted(data: &[Complex<f32>], rate: f32) -> Result<Vec<(f32, Complex<f32>)>, Error> {
    if data.is_empty() { return Ok(vec![]); }
    let cfg = sdr_fft_config_t { n: data.len(), input_format: SDR_FMT_C64, flags: SDR_FFT_SHIFT | SDR_FFT_NORM,
                                 device: 0, stream: std::ptr::null_mut() };
    let mut err = 0;
    let plan = unsafe { sdr_fft_create(&cfg, &mut err) };
    if plan.is_null() { return Err(Error(err)); }
    let mut vals = vec![Complex::new(0.0f32, 0.0); data.len()];
    let mut labels = vec![0.0f32; data.len()];
    let rc = unsafe { sdr_fft_exec(plan, data.as_ptr() as *const c_void, 1, vals.as_mut_ptr() as *mut f32) };
    unsafe { sdr_fft_destroy(plan) };
    check(rc)?;
    check(unsafe { sdr_fft_labels(data.len(), rate, 0, labels.as_mut_ptr()) })?;
    Ok(labels.into_iter().zip(vals.into_iter()).collect())
}

//! sdr_b200_sys.rs -- raw `extern "C"` bindings to libsdr_b200.so (include/sdr_b200.h).
//!
//! NOT COMPILED IN THIS REPOSITORY'S BUILD ENVIRONMENT: the image has no Rust toolchain (no cargo /
//! rustc).  This is the binding a maintainer of agrif/unnamed-rust-sdr would add as a `-sys` module; the
//! same ABI is exercised here from C++ (host/sdr.hpp, tests/cpp) and Python ctypes (sdr_b200/_ffi.py).
//! Link with: `println!("cargo:rustc-link-lib=dylib=sdr_b200");` in build.rs.
#![allow(non_camel_case_types, non_snake_case, dead_code)]
use libc::{c_char, c_double, c_float, c_int, c_long, c_uint, c_void, size_t};

pub const SDR_OK: c_int = 0;
pub const SDR_FMT_U8IQ: c_int = 0;
pub const SDR_FMT_C64: c_int = 1;
pub const SDR_FMT_F32: c_int = 2;
pub const SDR_FIR_STRICT_ORDER: c_uint = 1;
pub const SDR_FFT_SHIFT: c_uint = 1;
pub const SDR_FFT_NORM: c_uint = 2;
pub const SDR_FFT_RFFT: c_uint = 4;
/// sdr_pll_config_t.flags: atan2 / sin / cos evaluated in f64 and rounded to f32 (default: f32 routines within ~1 ulp)
pub const SDR_PLL_F64_MATH: c_uint = 2;
/// sdr_pfb_config_t.flags
pub const SDR_PFB_SHIFT: c_uint = 1;
pub const SDR_PFB_CHANNEL_MAJOR: c_uint = 2;
pub const SDR_PFB_GENERAL_KERNEL: c_uint = 4;
/// sdr_pfs_config_t.flags
pub const SDR_PFS_SHIFT: c_uint = 1;
pub const SDR_PFS_CHANNEL_MAJOR: c_uint = 2;
pub const SDR_PFS_GENERAL_KERNEL: c_uint = 4;
/// sdr_ddc_config_t.flags
pub const SDR_DDC_GENERAL_KERNEL: c_uint = 1;
/// sdr_psd_config_t.flags
pub const SDR_PSD_SHIFT: c_uint = 1;
pub const SDR_PSD_NORM: c_uint = 2;
pub const SDR_PSD_GENERAL_KERNEL: c_uint = 4;

pub enum sdr_fir_t {}
pub enum sdr_fft_t {}
pub enum sdr_pll_t {}
pub enum sdr_biquad_t {}
pub enum sdr_fm_t {}
pub enum sdr_window_fft_t {}
pub enum sdr_pfb_t {}
pub enum sdr_ddc_t {}
pub enum sdr_psd_t {}
pub enum sdr_fcfb_t {}
pub enum sdr_pfs_t {}
pub enum sdr_duc_t {}
pub enum sdr_fcsb_t {}
pub enum sdr_rrb_t {}
pub enum sdr_arb_t {}
pub enum sdr_tsync_t {}
pub enum sdr_csync_t {}
pub enum sdr_eq_t {}
pub enum sdr_vit_t {}
pub enum sdr_fsync_t {}
pub enum sdr_channelizer_t {}
/// same role as libsamplerate's SRC_STATE (src/resample.rs:12)
pub enum SDR_SRC_STATE {}

#[repr(C)]
pub struct sdr_fir_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub taps_complex: c_int,
    pub input_format: c_int,
    pub decimation: size_t,
    pub n_channels: size_t,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_fft_config_t {
    pub n: size_t,
    pub input_format: c_int,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct sdr_biquad_design_t {
    pub kind: c_int,
    pub p0: c_float,
    pub p1: c_float,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct sdr_pll_design_t {
    pub reference: c_float,
    pub gain: c_float,
    pub loopfilter: sdr_biquad_design_t,
    pub outputfilter: sdr_biquad_design_t,
    pub lockfilter: sdr_biquad_design_t,
}

#[repr(C)]
pub struct sdr_pll_config_t {
    pub designs: *const sdr_pll_design_t,
    pub n_designs: size_t,
    pub n_streams: size_t,
    pub rate: c_float,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_biquad_config_t {
    pub designs: *const sdr_biquad_design_t,
    pub n_designs: size_t,
    pub n_streams: size_t,
    pub rate: c_float,
    pub sample_complex: c_int,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_window_fft_config_t {
    pub window: size_t,
    pub hop: size_t,
    pub input_format: c_int,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_pfb_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_channels: size_t,
    pub decimation: size_t,
    pub input_format: c_int,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_pfs_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_channels: size_t,
    pub interpolation: size_t,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_ddc_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phase_inc: *const u64,
    pub n_channels: size_t,
    pub decimation: size_t,
    pub first_sample: u64,
    pub input_format: c_int,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_duc_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phase_inc: *const u64,
    pub n_channels: size_t,
    pub interpolation: size_t,
    pub first_sample: u64,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_psd_config_t {
    pub n: size_t,
    pub hop: size_t,
    pub average: size_t,
    pub window: *const c_float,
    pub input_format: c_int,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_fcfb_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phase_inc: *const u64,
    pub decimation: *const size_t,
    pub n_channels: size_t,
    pub first_sample: u64,
    pub input_format: c_int,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_fcsb_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phase_inc: *const u64,
    pub interpolation: *const size_t,
    pub n_channels: size_t,
    pub first_sample: u64,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_rrb_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub interpolation: *const size_t,
    pub decimation: *const size_t,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

/// whole + frac / 2^64 input frames
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct sdr_arb_time_t {
    pub whole: u64,
    pub frac: u64,
}

#[repr(C)]
pub struct sdr_arb_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phases: size_t,
    pub step: *const sdr_arb_time_t,
    pub first: *const sdr_arb_time_t,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct sdr_tsync_loop_t {
    pub kp: c_float,
    pub ki: c_float,
    pub err_max: c_float,
    pub max_dev: c_double,
}

#[repr(C)]
pub struct sdr_tsync_config_t {
    pub taps: *const c_float,
    pub n_taps: size_t,
    pub n_tap_sets: size_t,
    pub phases: size_t,
    pub period: *const sdr_arb_time_t,
    pub first: *const sdr_arb_time_t,
    pub loops: *const sdr_tsync_loop_t,
    pub n_loops: size_t,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct sdr_csync_loop_t {
    pub order: c_uint,
    pub kp: c_float,
    pub ki: c_float,
    pub err_max: c_float,
    pub max_freq: c_double,
}

#[repr(C)]
pub struct sdr_csync_config_t {
    pub loops: *const sdr_csync_loop_t,
    pub n_loops: size_t,
    pub phase: *const u64,
    pub freq: *const i64,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct sdr_eq_adapt_t {
    pub order: c_uint,
    pub mu: c_float,
    pub radius: c_float,
    pub err_max: c_float,
    pub cma_symbols: u64,
}

#[repr(C)]
pub struct sdr_eq_config_t {
    pub n_taps: size_t,
    pub taps: *const c_float,
    pub n_tap_sets: size_t,
    pub adapt: *const sdr_eq_adapt_t,
    pub n_adapt: size_t,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
pub struct sdr_vit_config_t {
    pub constraint: c_uint,
    pub gens: *const u32,
    pub n_gens: size_t,
    pub depth: size_t,
    pub scale: *const c_float,
    pub n_scales: size_t,
    pub zero_start: c_int,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

pub const SDR_FSYNC_SEARCH: u32 = 0;
pub const SDR_FSYNC_VERIFY: u32 = 1;
pub const SDR_FSYNC_LOCK: u32 = 2;
pub const SDR_FSYNC_HIT: u16 = 1;
pub const SDR_FSYNC_VERIFY_PASS: u16 = 2;
pub const SDR_FSYNC_VERIFY_FAIL: u16 = 3;
pub const SDR_FSYNC_LOCK_PASS: u16 = 4;
pub const SDR_FSYNC_LOCK_MISS: u16 = 5;
pub const SDR_FSYNC_LOCK_LOST: u16 = 6;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct sdr_fsync_params_t {
    pub period: u32,
    pub order: u32,
    pub thresh_search: c_float,
    pub thresh_check: c_float,
    pub verify: u32,
    pub max_miss: u32,
    pub window: u32,
}

#[repr(C)]
pub struct sdr_fsync_config_t {
    pub word_len: size_t,
    pub words: *const c_float,
    pub n_words: size_t,
    pub params: *const sdr_fsync_params_t,
    pub n_params: size_t,
    pub n_channels: size_t,
    pub device: c_int,
    pub stream: *mut c_void,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct sdr_fsync_record_t {
    pub pos: u64,
    pub out_index: u64,
    pub corr: [c_float; 2],
    pub rho: c_float,
    pub rot: u16,
    pub kind: u16,
}

#[repr(C)]
#[derive(Clone, Copy, Default, Debug)]
pub struct sdr_fsync_state_t {
    pub state: u32,
    pub count: u32,
    pub pos: u64,
    pub rot: u32,
    pub pad: u32,
    pub consumed: u64,
    pub payload: u64,
}

#[repr(C)]
pub struct sdr_fm_config_t {
    pub n_stations: size_t,
    pub rate: c_float,
    pub pilot: c_float,
    pub flags: c_uint,
    pub device: c_int,
    pub stream: *mut c_void,
}

/// identical layout to libsamplerate's SRC_DATA as built at src/resample.rs:49-58
#[repr(C)]
pub struct SDR_SRC_DATA {
    pub data_in: *const c_float,
    pub data_out: *mut c_float,
    pub input_frames: c_long,
    pub output_frames: c_long,
    pub input_frames_used: c_long,
    pub output_frames_gen: c_long,
    pub end_of_input: c_int,
    pub src_ratio: c_double,
}

extern "C" {
    pub fn sdr_strerror(code: c_int) -> *const c_char;
    pub fn sdr_device_count() -> c_int;

    pub fn sdr_unpack_u8iq(iq: *const u8, n_samples: size_t, out_c64: *mut c_float, device: c_int) -> c_int;

    pub fn sdr_fir_create(cfg: *const sdr_fir_config_t, err: *mut c_int) -> *mut sdr_fir_t;
    pub fn sdr_fir_destroy(f: *mut sdr_fir_t);
    pub fn sdr_fir_reset(f: *mut sdr_fir_t) -> c_int;
    pub fn sdr_fir_clone(f: *const sdr_fir_t, err: *mut c_int) -> *mut sdr_fir_t;
    pub fn sdr_fir_output_count(f: *const sdr_fir_t, n_in: size_t) -> size_t;
    pub fn sdr_fir_process(f: *mut sdr_fir_t, input: *const c_void, n_in: size_t, in_stride: size_t,
                           output: *mut c_void, out_cap: size_t, out_stride: size_t,
                           n_used: *mut size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_decimate_wait(rate_in: c_float, rate_out: c_float) -> size_t;

    pub fn sdr_fft_create(cfg: *const sdr_fft_config_t, err: *mut c_int) -> *mut sdr_fft_t;
    pub fn sdr_fft_destroy(p: *mut sdr_fft_t);
    pub fn sdr_fft_output_len(p: *const sdr_fft_t) -> size_t;
    pub fn sdr_fft_exec(p: *mut sdr_fft_t, input: *const c_void, batches: size_t, out_c64: *mut c_float) -> c_int;
    pub fn sdr_fft_labels(n: size_t, rate: c_float, rfft: c_int, labels: *mut c_float) -> c_int;

    pub fn sdr_pll_create(cfg: *const sdr_pll_config_t, err: *mut c_int) -> *mut sdr_pll_t;
    pub fn sdr_pll_destroy(p: *mut sdr_pll_t);
    pub fn sdr_pll_reset(p: *mut sdr_pll_t) -> c_int;
    pub fn sdr_pll_clone(p: *const sdr_pll_t, err: *mut c_int) -> *mut sdr_pll_t;
    pub fn sdr_pll_process(p: *mut sdr_pll_t, in_c64: *const c_float, n: size_t, in_stride: size_t,
                           out: *mut c_float, locked: *mut u8, out_stride: size_t) -> c_int;
    pub fn sdr_pll_get_state(p: *mut sdr_pll_t, idx: size_t, nphase: *mut c_float, re: *mut c_float, im: *mut c_float) -> c_int;

    // Biquad<f32, A> as a stream filter (src/filter/biquad.rs:40-56)
    pub fn sdr_biquad_create(cfg: *const sdr_biquad_config_t, err: *mut c_int) -> *mut sdr_biquad_t;
    pub fn sdr_biquad_destroy(b: *mut sdr_biquad_t);
    pub fn sdr_biquad_reset(b: *mut sdr_biquad_t) -> c_int;
    pub fn sdr_biquad_clone(b: *const sdr_biquad_t, err: *mut c_int) -> *mut sdr_biquad_t;
    pub fn sdr_biquad_process(b: *mut sdr_biquad_t, input: *const c_float, n: size_t, in_stride: size_t,
                              output: *mut c_float, out_stride: size_t) -> c_int;

    // src/main.rs:62-71 (pilot Pll + stereo decode) and src/main.rs:32-81 (the whole FM stereo receiver)
    pub fn sdr_pll_stereo_decode(p: *mut sdr_pll_t, v: *const c_float, n: size_t, in_stride: size_t,
                                 out_mono_diff: *mut c_float, out_stride: size_t) -> c_int;
    pub fn sdr_fm_create(cfg: *const sdr_fm_config_t, err: *mut c_int) -> *mut sdr_fm_t;
    pub fn sdr_fm_destroy(f: *mut sdr_fm_t);
    pub fn sdr_fm_reset(f: *mut sdr_fm_t) -> c_int;
    pub fn sdr_fm_output_rate(f: *const sdr_fm_t) -> c_float;
    pub fn sdr_fm_max_output(f: *const sdr_fm_t, n: size_t) -> size_t;
    pub fn sdr_fm_process(f: *mut sdr_fm_t, iq: *const u8, n: size_t, in_stride: size_t, out: *mut c_float,
                          out_cap: size_t, out_stride: size_t, n_out: *mut size_t, end_of_input: c_int) -> c_int;

    // examples/live.rs:30-39: window(duration).decimate(fps).map(fft::fft)
    pub fn sdr_window_fft_create(cfg: *const sdr_window_fft_config_t, err: *mut c_int) -> *mut sdr_window_fft_t;
    pub fn sdr_window_fft_destroy(h: *mut sdr_window_fft_t);
    pub fn sdr_window_fft_reset(h: *mut sdr_window_fft_t) -> c_int;
    pub fn sdr_window_fft_size(h: *const sdr_window_fft_t) -> size_t;
    pub fn sdr_window_fft_output_count(h: *const sdr_window_fft_t, n_in: size_t) -> size_t;
    pub fn sdr_window_fft_process(h: *mut sdr_window_fft_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float,
                                  out_cap: size_t, n_windows: *mut size_t) -> c_int;

    // polyphase filter bank: M x (Fir(h e^{+2 pi i k n / M}) + Decimate(D)) in one pass
    pub fn sdr_pfb_create(cfg: *const sdr_pfb_config_t, err: *mut c_int) -> *mut sdr_pfb_t;
    pub fn sdr_pfb_destroy(h: *mut sdr_pfb_t);
    pub fn sdr_pfb_reset(h: *mut sdr_pfb_t) -> c_int;
    pub fn sdr_pfb_clone(h: *const sdr_pfb_t, err: *mut c_int) -> *mut sdr_pfb_t;
    pub fn sdr_pfb_output_count(h: *const sdr_pfb_t, n_in: size_t) -> size_t;
    pub fn sdr_pfb_process(h: *mut sdr_pfb_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float, out_cap: size_t,
                           out_stride: size_t, n_frames: *mut size_t) -> c_int;
    pub fn sdr_pfb_process_dev(h: *mut sdr_pfb_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float,
                               out_cap: size_t, out_stride: size_t, n_frames: *mut size_t) -> c_int;

    // polyphase synthesis bank: M channel streams -> one stream at D samples per frame (the inverse of sdr_pfb)
    pub fn sdr_pfs_create(cfg: *const sdr_pfs_config_t, err: *mut c_int) -> *mut sdr_pfs_t;
    pub fn sdr_pfs_destroy(h: *mut sdr_pfs_t);
    pub fn sdr_pfs_reset(h: *mut sdr_pfs_t) -> c_int;
    pub fn sdr_pfs_clone(h: *const sdr_pfs_t, err: *mut c_int) -> *mut sdr_pfs_t;
    pub fn sdr_pfs_output_count(h: *const sdr_pfs_t, n_frames: size_t) -> size_t;
    pub fn sdr_pfs_process(h: *mut sdr_pfs_t, in_c64: *const c_float, n_frames: size_t, in_stride: size_t,
                           out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_pfs_process_dev(h: *mut sdr_pfs_t, in_c64: *const c_float, n_frames: size_t, in_stride: size_t,
                               out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;

    // down-converter bank: C x (64-bit NCO mixer + Fir(h_k) + Decimate(D)) in one pass
    pub fn sdr_ddc_phase_increment(freq: f64, rate: f64) -> u64;
    pub fn sdr_ddc_create(cfg: *const sdr_ddc_config_t, err: *mut c_int) -> *mut sdr_ddc_t;
    pub fn sdr_ddc_destroy(h: *mut sdr_ddc_t);
    pub fn sdr_ddc_reset(h: *mut sdr_ddc_t) -> c_int;
    pub fn sdr_ddc_clone(h: *const sdr_ddc_t, err: *mut c_int) -> *mut sdr_ddc_t;
    pub fn sdr_ddc_output_count(h: *const sdr_ddc_t, n_in: size_t) -> size_t;
    pub fn sdr_ddc_process(h: *mut sdr_ddc_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float, out_cap: size_t,
                           out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_ddc_process_dev(h: *mut sdr_ddc_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float,
                               out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_ddc_last_path(h: *const sdr_ddc_t) -> c_int;

    // up-converter bank: C x (zero-stuff(I) + Fir(h_k) + 64-bit NCO mix up), summed into one stream
    pub fn sdr_duc_create(cfg: *const sdr_duc_config_t, err: *mut c_int) -> *mut sdr_duc_t;
    pub fn sdr_duc_destroy(h: *mut sdr_duc_t);
    pub fn sdr_duc_reset(h: *mut sdr_duc_t) -> c_int;
    pub fn sdr_duc_clone(h: *const sdr_duc_t, err: *mut c_int) -> *mut sdr_duc_t;
    pub fn sdr_duc_output_count(h: *const sdr_duc_t, n_frames: size_t) -> size_t;
    pub fn sdr_duc_process(h: *mut sdr_duc_t, in_c64: *const c_float, n_frames: size_t, in_stride: size_t,
                           out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_duc_process_dev(h: *mut sdr_duc_t, in_c64: *const c_float, n_frames: size_t, in_stride: size_t,
                               out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_psd_create(cfg: *const sdr_psd_config_t, err: *mut c_int) -> *mut sdr_psd_t;
    pub fn sdr_psd_destroy(h: *mut sdr_psd_t);
    pub fn sdr_psd_reset(h: *mut sdr_psd_t) -> c_int;
    pub fn sdr_psd_clone(h: *const sdr_psd_t, err: *mut c_int) -> *mut sdr_psd_t;
    pub fn sdr_psd_output_count(h: *const sdr_psd_t, n_in: size_t) -> size_t;
    pub fn sdr_psd_process(h: *mut sdr_psd_t, input: *const c_void, n_in: size_t, out: *mut c_float, out_cap: size_t,
                           out_stride: size_t, n_spectra: *mut size_t) -> c_int;
    pub fn sdr_psd_process_dev(h: *mut sdr_psd_t, input: *const c_void, n_in: size_t, out: *mut c_float,
                               out_cap: size_t, out_stride: size_t, n_spectra: *mut size_t) -> c_int;
    pub fn sdr_psd_last_path(h: *const sdr_psd_t) -> c_int;
    pub fn sdr_fcfb_geometry(n_taps: size_t, decimation: *const size_t, n_channels: size_t, n_fft: *mut size_t,
                             hop: *mut size_t) -> c_int;
    pub fn sdr_fcfb_create(cfg: *const sdr_fcfb_config_t, err: *mut c_int) -> *mut sdr_fcfb_t;
    pub fn sdr_fcfb_destroy(h: *mut sdr_fcfb_t);
    pub fn sdr_fcfb_reset(h: *mut sdr_fcfb_t) -> c_int;
    pub fn sdr_fcfb_clone(h: *const sdr_fcfb_t, err: *mut c_int) -> *mut sdr_fcfb_t;
    pub fn sdr_fcfb_output_count(h: *const sdr_fcfb_t, n_in: size_t, counts: *mut size_t) -> c_int;
    pub fn sdr_fcfb_process(h: *mut sdr_fcfb_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float,
                            out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_fcfb_process_dev(h: *mut sdr_fcfb_t, input: *const c_void, n_in: size_t, out_c64: *mut c_float,
                                out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_fcsb_create(cfg: *const sdr_fcsb_config_t, err: *mut c_int) -> *mut sdr_fcsb_t;
    pub fn sdr_fcsb_destroy(h: *mut sdr_fcsb_t);
    pub fn sdr_fcsb_reset(h: *mut sdr_fcsb_t) -> c_int;
    pub fn sdr_fcsb_clone(h: *const sdr_fcsb_t, err: *mut c_int) -> *mut sdr_fcsb_t;
    pub fn sdr_fcsb_output_count(h: *const sdr_fcsb_t, n_time: size_t) -> size_t;
    pub fn sdr_fcsb_process(h: *mut sdr_fcsb_t, in_c64: *const c_float, n_time: size_t, in_stride: size_t,
                            out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_fcsb_process_dev(h: *mut sdr_fcsb_t, in_c64: *const c_float, n_time: size_t, in_stride: size_t,
                                out_c64: *mut c_float, out_cap: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_rrb_create(cfg: *const sdr_rrb_config_t, err: *mut c_int) -> *mut sdr_rrb_t;
    pub fn sdr_rrb_destroy(h: *mut sdr_rrb_t);
    pub fn sdr_rrb_reset(h: *mut sdr_rrb_t) -> c_int;
    pub fn sdr_rrb_clone(h: *const sdr_rrb_t, err: *mut c_int) -> *mut sdr_rrb_t;
    pub fn sdr_rrb_output_count(h: *const sdr_rrb_t, n_in: *const size_t, counts: *mut size_t) -> c_int;
    pub fn sdr_rrb_process(h: *mut sdr_rrb_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                           out_c64: *mut c_float, out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_rrb_process_dev(h: *mut sdr_rrb_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                               out_c64: *mut c_float, out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_arb_step(rate_in: c_double, rate_out: c_double, step: *mut sdr_arb_time_t) -> c_int;
    pub fn sdr_arb_create(cfg: *const sdr_arb_config_t, err: *mut c_int) -> *mut sdr_arb_t;
    pub fn sdr_arb_destroy(h: *mut sdr_arb_t);
    pub fn sdr_arb_reset(h: *mut sdr_arb_t) -> c_int;
    pub fn sdr_arb_clone(h: *const sdr_arb_t, err: *mut c_int) -> *mut sdr_arb_t;
    pub fn sdr_arb_set_steps(h: *mut sdr_arb_t, steps: *const sdr_arb_time_t) -> c_int;
    pub fn sdr_arb_output_count(h: *const sdr_arb_t, n_in: *const size_t, counts: *mut size_t) -> c_int;
    pub fn sdr_arb_process(h: *mut sdr_arb_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                           out_c64: *mut c_float, out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_arb_process_dev(h: *mut sdr_arb_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                               out_c64: *mut c_float, out_cap: size_t, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_tsync_loop_design(bn_t: c_double, zeta: c_double, ted_gain: c_double, period_frames: c_double,
                                 kp: *mut c_float, ki: *mut c_float) -> c_int;
    pub fn sdr_tsync_create(cfg: *const sdr_tsync_config_t, err: *mut c_int) -> *mut sdr_tsync_t;
    pub fn sdr_tsync_destroy(h: *mut sdr_tsync_t);
    pub fn sdr_tsync_reset(h: *mut sdr_tsync_t) -> c_int;
    pub fn sdr_tsync_clone(h: *const sdr_tsync_t, err: *mut c_int) -> *mut sdr_tsync_t;
    pub fn sdr_tsync_max_output(h: *const sdr_tsync_t, n_in: *const size_t, caps: *mut size_t) -> c_int;
    pub fn sdr_tsync_process(h: *mut sdr_tsync_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                             sym_c64: *mut c_float, pos: *mut sdr_arb_time_t, err: *mut c_float, out_cap: size_t,
                             out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_tsync_process_dev(h: *mut sdr_tsync_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                                 sym_c64: *mut c_float, pos: *mut sdr_arb_time_t, err: *mut c_float, out_cap: size_t,
                                 out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_tsync_get_state(h: *mut sdr_tsync_t, channel: size_t, next: *mut sdr_arb_time_t, v: *mut i64) -> c_int;
    pub fn sdr_csync_create(cfg: *const sdr_csync_config_t, err: *mut c_int) -> *mut sdr_csync_t;
    pub fn sdr_csync_destroy(h: *mut sdr_csync_t);
    pub fn sdr_csync_reset(h: *mut sdr_csync_t) -> c_int;
    pub fn sdr_csync_clone(h: *const sdr_csync_t, err: *mut c_int) -> *mut sdr_csync_t;
    pub fn sdr_csync_process(h: *mut sdr_csync_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                             out_c64: *mut c_float, phase: *mut u64, err: *mut c_float, out_stride: size_t) -> c_int;
    pub fn sdr_csync_process_dev(h: *mut sdr_csync_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                                 out_c64: *mut c_float, phase: *mut u64, err: *mut c_float, out_stride: size_t)
                                 -> c_int;
    pub fn sdr_csync_get_state(h: *mut sdr_csync_t, channel: size_t, phase: *mut u64, freq: *mut i64) -> c_int;
    pub fn sdr_eq_create(cfg: *const sdr_eq_config_t, err: *mut c_int) -> *mut sdr_eq_t;
    pub fn sdr_eq_destroy(h: *mut sdr_eq_t);
    pub fn sdr_eq_reset(h: *mut sdr_eq_t) -> c_int;
    pub fn sdr_eq_clone(h: *const sdr_eq_t, err: *mut c_int) -> *mut sdr_eq_t;
    pub fn sdr_eq_process(h: *mut sdr_eq_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                          out_c64: *mut c_float, err_c64: *mut c_float, out_stride: size_t) -> c_int;
    pub fn sdr_eq_process_dev(h: *mut sdr_eq_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                              out_c64: *mut c_float, err_c64: *mut c_float, out_stride: size_t) -> c_int;
    pub fn sdr_eq_get_taps(h: *mut sdr_eq_t, channel: size_t, taps_c64: *mut c_float) -> c_int;
    pub fn sdr_vit_create(cfg: *const sdr_vit_config_t, err: *mut c_int) -> *mut sdr_vit_t;
    pub fn sdr_vit_destroy(h: *mut sdr_vit_t);
    pub fn sdr_vit_reset(h: *mut sdr_vit_t) -> c_int;
    pub fn sdr_vit_clone(h: *const sdr_vit_t, err: *mut c_int) -> *mut sdr_vit_t;
    pub fn sdr_vit_output_count(h: *const sdr_vit_t, n_in: *const size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_vit_process(h: *mut sdr_vit_t, input: *const c_float, n_in: *const size_t, in_stride: size_t,
                           out: *mut u8, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_vit_process_dev(h: *mut sdr_vit_t, input: *const c_float, n_in: *const size_t, in_stride: size_t,
                               out: *mut u8, out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_vit_finish(h: *mut sdr_vit_t, which: *const u8, terminated: c_int, out: *mut u8, out_stride: size_t,
                          n_out: *mut size_t) -> c_int;
    pub fn sdr_vit_finish_dev(h: *mut sdr_vit_t, which: *const u8, terminated: c_int, out: *mut u8,
                              out_stride: size_t, n_out: *mut size_t) -> c_int;
    pub fn sdr_fsync_create(cfg: *const sdr_fsync_config_t, err: *mut c_int) -> *mut sdr_fsync_t;
    pub fn sdr_fsync_destroy(h: *mut sdr_fsync_t);
    pub fn sdr_fsync_reset(h: *mut sdr_fsync_t) -> c_int;
    pub fn sdr_fsync_clone(h: *const sdr_fsync_t, err: *mut c_int) -> *mut sdr_fsync_t;
    pub fn sdr_fsync_max_output(h: *const sdr_fsync_t, n_in: *const size_t, pay_caps: *mut size_t,
                                rec_caps: *mut size_t) -> c_int;
    pub fn sdr_fsync_process(h: *mut sdr_fsync_t, in_c64: *const c_float, n_in: *const size_t, in_stride: size_t,
                             out_c64: *mut c_float, out_cap: size_t, out_stride: size_t, n_out: *mut size_t,
                             recs: *mut sdr_fsync_record_t, rec_cap: size_t, rec_stride: size_t,
                             n_rec: *mut size_t) -> c_int;
    pub fn sdr_fsync_process_dev(h: *mut sdr_fsync_t, in_c64: *const c_float, n_in: *const size_t,
                                 in_stride: size_t, out_c64: *mut c_float, out_cap: size_t, out_stride: size_t,
                                 n_out: *mut size_t, recs: *mut sdr_fsync_record_t, rec_cap: size_t,
                                 rec_stride: size_t, n_rec: *mut size_t) -> c_int;
    pub fn sdr_fsync_get_state(h: *mut sdr_fsync_t, channel: size_t, state: *mut sdr_fsync_state_t) -> c_int;

    // drop-in for libsamplerate_sys::{src_new, src_process, ...} used by src/resample.rs
    pub fn sdr_src_new(converter_type: c_int, channels: c_int, error: *mut c_int) -> *mut SDR_SRC_STATE;
    pub fn sdr_src_delete(s: *mut SDR_SRC_STATE) -> *mut SDR_SRC_STATE;
    pub fn sdr_src_process(s: *mut SDR_SRC_STATE, data: *mut SDR_SRC_DATA) -> c_int;
    pub fn sdr_src_reset(s: *mut SDR_SRC_STATE) -> c_int;
    pub fn sdr_src_clone(s: *mut SDR_SRC_STATE, error: *mut c_int) -> *mut SDR_SRC_STATE;
    pub fn sdr_src_set_ratio(s: *mut SDR_SRC_STATE, new_ratio: c_double) -> c_int;
    pub fn sdr_src_get_channels(s: *mut SDR_SRC_STATE) -> c_int;
    pub fn sdr_src_history_frames(s: *mut SDR_SRC_STATE) -> c_long;
    pub fn sdr_src_set_exact(s: *mut SDR_SRC_STATE, exact: c_int) -> c_int;
    pub fn sdr_src_strerror(error: c_int) -> *const c_char;
    pub fn sdr_src_get_name(converter_type: c_int) -> *const c_char;
    pub fn sdr_src_get_description(converter_type: c_int) -> *const c_char;
    pub fn sdr_src_get_version() -> *const c_char;
}

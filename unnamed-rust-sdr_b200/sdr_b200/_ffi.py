"""ctypes binding of include/sdr_b200.h (libsdr_b200.so).  No fallback: if the CUDA library is not
built or no CUDA device is present, loading / constructing fails loudly."""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_PKG), "lib", "libsdr_b200.so")

FMT_U8IQ, FMT_C64, FMT_F32 = 0, 1, 2
FIR_STRICT_ORDER, FIR_NO_TENSOR, FIR_NO_TCGEN05, FIR_PLANAR, FIR_SPLIT2 = 1, 2, 4, 8, 16
FFT_SHIFT, FFT_NORM, FFT_RFFT = 1, 2, 4
PLL_FAST_MATH = 1
PLL_F64_MATH = 2
PLL_GENERAL_KERNEL = 4
PFB_SHIFT, PFB_CHANNEL_MAJOR, PFB_GENERAL_KERNEL = 1, 2, 4
PFS_SHIFT, PFS_CHANNEL_MAJOR, PFS_GENERAL_KERNEL = 1, 2, 4
DDC_GENERAL_KERNEL = 1
PSD_SHIFT, PSD_NORM, PSD_GENERAL_KERNEL = 1, 2, 4
BQ_IDENTITY, BQ_LOWPASS, BQ_HIGHPASS, BQ_BANDPASS, BQ_NOTCH, BQ_LR = range(6)
SRC_SINC_BEST_QUALITY, SRC_SINC_MEDIUM_QUALITY, SRC_SINC_FASTEST, SRC_ZERO_ORDER_HOLD, SRC_LINEAR = range(5)

vp, sz, f32, i32 = C.c_void_p, C.c_size_t, C.c_float, C.c_int


class FirConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("taps_complex", i32), ("input_format", i32),
                ("decimation", sz), ("n_channels", sz), ("flags", C.c_uint), ("device", i32), ("stream", vp)]


class FftConfig(C.Structure):
    _fields_ = [("n", sz), ("input_format", i32), ("flags", C.c_uint), ("device", i32), ("stream", vp)]


class BiquadDesign(C.Structure):
    _fields_ = [("kind", i32), ("p0", f32), ("p1", f32)]


class PllDesign(C.Structure):
    _fields_ = [("reference", f32), ("gain", f32), ("loopfilter", BiquadDesign),
                ("outputfilter", BiquadDesign), ("lockfilter", BiquadDesign)]


class PllConfig(C.Structure):
    _fields_ = [("designs", vp), ("n_designs", sz), ("n_streams", sz), ("rate", f32),
                ("flags", C.c_uint), ("device", i32), ("stream", vp)]


class BiquadConfig(C.Structure):
    _fields_ = [("designs", vp), ("n_designs", sz), ("n_streams", sz), ("rate", f32),
                ("sample_complex", i32), ("device", i32), ("stream", vp)]


class FmConfig(C.Structure):
    _fields_ = [("n_stations", sz), ("rate", f32), ("pilot", f32), ("flags", C.c_uint), ("device", i32),
                ("stream", vp)]


class WindowFftConfig(C.Structure):
    _fields_ = [("window", sz), ("hop", sz), ("input_format", i32), ("flags", C.c_uint), ("device", i32), ("stream", vp)]


class PfbConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_channels", sz), ("decimation", sz), ("input_format", i32),
                ("flags", C.c_uint), ("device", i32), ("stream", vp)]


class DdcConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phase_inc", vp), ("n_channels", sz),
                ("decimation", sz), ("first_sample", C.c_uint64), ("input_format", i32), ("flags", C.c_uint),
                ("device", i32), ("stream", vp)]


class PsdConfig(C.Structure):
    _fields_ = [("n", sz), ("hop", sz), ("average", sz), ("window", vp), ("input_format", i32), ("flags", C.c_uint),
                ("device", i32), ("stream", vp)]


class FcfbConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phase_inc", vp), ("decimation", vp),
                ("n_channels", sz), ("first_sample", C.c_uint64), ("input_format", i32), ("device", i32),
                ("stream", vp)]


class PfsConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_channels", sz), ("interpolation", sz), ("flags", C.c_uint),
                ("device", i32), ("stream", vp)]


class DucConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phase_inc", vp), ("n_channels", sz),
                ("interpolation", sz), ("first_sample", C.c_uint64), ("flags", C.c_uint), ("device", i32),
                ("stream", vp)]


class FcsbConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phase_inc", vp), ("interpolation", vp),
                ("n_channels", sz), ("first_sample", C.c_uint64), ("device", i32), ("stream", vp)]


class RrbConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("interpolation", vp), ("decimation", vp),
                ("n_channels", sz), ("device", i32), ("stream", vp)]


class ArbTime(C.Structure):
    _fields_ = [("whole", C.c_uint64), ("frac", C.c_uint64)]


class ArbConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phases", sz), ("step", vp), ("first", vp),
                ("n_channels", sz), ("device", i32), ("stream", vp)]


class TsyncLoop(C.Structure):
    _fields_ = [("kp", C.c_float), ("ki", C.c_float), ("err_max", C.c_float), ("max_dev", C.c_double)]


class TsyncConfig(C.Structure):
    _fields_ = [("taps", vp), ("n_taps", sz), ("n_tap_sets", sz), ("phases", sz), ("period", vp), ("first", vp),
                ("loops", vp), ("n_loops", sz), ("n_channels", sz), ("device", i32), ("stream", vp)]


class CsyncLoop(C.Structure):
    _fields_ = [("order", C.c_uint), ("kp", C.c_float), ("ki", C.c_float), ("err_max", C.c_float),
                ("max_freq", C.c_double)]


class CsyncConfig(C.Structure):
    _fields_ = [("loops", vp), ("n_loops", sz), ("phase", vp), ("freq", vp), ("n_channels", sz), ("device", i32),
                ("stream", vp)]


class EqAdapt(C.Structure):
    _fields_ = [("order", C.c_uint), ("mu", C.c_float), ("radius", C.c_float), ("err_max", C.c_float),
                ("cma_symbols", C.c_uint64)]


class EqConfig(C.Structure):
    _fields_ = [("n_taps", sz), ("taps", vp), ("n_tap_sets", sz), ("adapt", vp), ("n_adapt", sz), ("n_channels", sz),
                ("device", i32), ("stream", vp)]


class VitConfig(C.Structure):
    _fields_ = [("constraint", C.c_uint), ("gens", vp), ("n_gens", sz), ("depth", sz), ("scale", vp), ("n_scales", sz),
                ("zero_start", i32), ("n_channels", sz), ("device", i32), ("stream", vp)]


class FsyncParams(C.Structure):
    _fields_ = [("period", C.c_uint32), ("order", C.c_uint32), ("thresh_search", C.c_float),
                ("thresh_check", C.c_float), ("verify", C.c_uint32), ("max_miss", C.c_uint32), ("window", C.c_uint32)]


class FsyncConfig(C.Structure):
    _fields_ = [("word_len", sz), ("words", vp), ("n_words", sz), ("params", vp), ("n_params", sz),
                ("n_channels", sz), ("device", i32), ("stream", vp)]


class FsyncState(C.Structure):
    _fields_ = [("state", C.c_uint32), ("count", C.c_uint32), ("pos", C.c_uint64), ("rot", C.c_uint32),
                ("pad", C.c_uint32), ("consumed", C.c_uint64), ("payload", C.c_uint64)]


class SrcData(C.Structure):
    _fields_ = [("data_in", vp), ("data_out", vp), ("input_frames", C.c_long), ("output_frames", C.c_long),
                ("input_frames_used", C.c_long), ("output_frames_gen", C.c_long),
                ("end_of_input", i32), ("src_ratio", C.c_double)]


# name -> (restype, argtypes): every symbol include/sdr_b200.h declares
PROTOTYPES = {
    "sdr_strerror": (C.c_char_p, [i32]),
    "sdr_abi_version": (i32, []),
    "sdr_device_count": (i32, []),
    "sdr_device_info": (i32, [i32, C.c_char_p, sz]),
    "sdr_unpack_u8iq": (i32, [vp, sz, vp, i32]),
    "sdr_unpack_u8iq_dev": (i32, [vp, sz, vp, i32, vp]),
    "sdr_fir_create": (vp, [C.POINTER(FirConfig), C.POINTER(i32)]),
    "sdr_fir_destroy": (None, [vp]),
    "sdr_fir_reset": (i32, [vp]),
    "sdr_fir_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_fir_output_count": (sz, [vp, sz]),
    "sdr_fir_process": (i32, [vp, vp, sz, sz, vp, sz, sz, C.POINTER(sz), C.POINTER(sz)]),
    "sdr_fir_process_dev": (i32, [vp, vp, sz, sz, vp, sz, sz, C.POINTER(sz), C.POINTER(sz)]),
    "sdr_fir_last_path": (i32, [vp]),
    "sdr_decimate_wait": (sz, [f32, f32]),
    "sdr_duration_samples": (sz, [f32, f32]),
    "sdr_block_samples": (sz, [f32, f32]),
    "sdr_fft_create": (vp, [C.POINTER(FftConfig), C.POINTER(i32)]),
    "sdr_fft_destroy": (None, [vp]),
    "sdr_fft_output_len": (sz, [vp]),
    "sdr_fft_exec": (i32, [vp, vp, sz, vp]),
    "sdr_fft_exec_dev": (i32, [vp, vp, sz, vp]),
    "sdr_fft_labels": (i32, [sz, f32, i32, vp]),
    "sdr_biquad_design": (i32, [C.POINTER(BiquadDesign), f32, vp]),
    "sdr_pll_create": (vp, [C.POINTER(PllConfig), C.POINTER(i32)]),
    "sdr_pll_destroy": (None, [vp]),
    "sdr_pll_reset": (i32, [vp]),
    "sdr_pll_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_pll_process": (i32, [vp, vp, sz, sz, vp, vp, sz]),
    "sdr_pll_process_dev": (i32, [vp, vp, sz, sz, vp, vp, sz]),
    "sdr_pll_stereo_decode": (i32, [vp, vp, sz, sz, vp, sz]),
    "sdr_pll_stereo_decode_dev": (i32, [vp, vp, sz, sz, vp, sz]),
    "sdr_pll_get_state": (i32, [vp, sz, C.POINTER(f32), C.POINTER(f32), C.POINTER(f32)]),
    "sdr_window_fft_create": (vp, [C.POINTER(WindowFftConfig), C.POINTER(i32)]),
    "sdr_window_fft_destroy": (None, [vp]),
    "sdr_window_fft_reset": (i32, [vp]),
    "sdr_window_fft_size": (sz, [vp]),
    "sdr_window_fft_output_count": (sz, [vp, sz]),
    "sdr_window_fft_process": (i32, [vp, vp, sz, vp, sz, C.POINTER(sz)]),
    "sdr_window_fft_process_dev": (i32, [vp, vp, sz, vp, sz, C.POINTER(sz)]),
    "sdr_pfb_create": (vp, [C.POINTER(PfbConfig), C.POINTER(i32)]),
    "sdr_pfb_destroy": (None, [vp]),
    "sdr_pfb_reset": (i32, [vp]),
    "sdr_pfb_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_pfb_output_count": (sz, [vp, sz]),
    "sdr_pfb_process": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_pfb_process_dev": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_pfs_create": (vp, [C.POINTER(PfsConfig), C.POINTER(i32)]),
    "sdr_pfs_destroy": (None, [vp]),
    "sdr_pfs_reset": (i32, [vp]),
    "sdr_pfs_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_pfs_output_count": (sz, [vp, sz]),
    "sdr_pfs_process": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_pfs_process_dev": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_duc_create": (vp, [C.POINTER(DucConfig), C.POINTER(i32)]),
    "sdr_duc_destroy": (None, [vp]),
    "sdr_duc_reset": (i32, [vp]),
    "sdr_duc_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_duc_output_count": (sz, [vp, sz]),
    "sdr_duc_process": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_duc_process_dev": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_ddc_phase_increment": (C.c_uint64, [C.c_double, C.c_double]),
    "sdr_ddc_create": (vp, [C.POINTER(DdcConfig), C.POINTER(i32)]),
    "sdr_ddc_destroy": (None, [vp]),
    "sdr_ddc_reset": (i32, [vp]),
    "sdr_ddc_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_ddc_output_count": (sz, [vp, sz]),
    "sdr_ddc_process": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_ddc_process_dev": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_ddc_last_path": (i32, [vp]),
    "sdr_psd_create": (vp, [C.POINTER(PsdConfig), C.POINTER(i32)]),
    "sdr_psd_destroy": (None, [vp]),
    "sdr_psd_reset": (i32, [vp]),
    "sdr_psd_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_psd_output_count": (sz, [vp, sz]),
    "sdr_psd_process": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_psd_process_dev": (i32, [vp, vp, sz, vp, sz, sz, C.POINTER(sz)]),
    "sdr_psd_last_path": (i32, [vp]),
    "sdr_fcfb_geometry": (i32, [sz, vp, sz, C.POINTER(sz), C.POINTER(sz)]),
    "sdr_fcfb_create": (vp, [C.POINTER(FcfbConfig), C.POINTER(i32)]),
    "sdr_fcfb_destroy": (None, [vp]),
    "sdr_fcfb_reset": (i32, [vp]),
    "sdr_fcfb_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_fcfb_output_count": (i32, [vp, sz, vp]),
    "sdr_fcfb_process": (i32, [vp, vp, sz, vp, sz, sz, vp]),
    "sdr_fcfb_process_dev": (i32, [vp, vp, sz, vp, sz, sz, vp]),
    "sdr_fcsb_create": (vp, [C.POINTER(FcsbConfig), C.POINTER(i32)]),
    "sdr_fcsb_destroy": (None, [vp]),
    "sdr_fcsb_reset": (i32, [vp]),
    "sdr_fcsb_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_fcsb_output_count": (sz, [vp, sz]),
    "sdr_fcsb_process": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_fcsb_process_dev": (i32, [vp, vp, sz, sz, vp, sz, C.POINTER(sz)]),
    "sdr_rrb_create": (vp, [C.POINTER(RrbConfig), C.POINTER(i32)]),
    "sdr_rrb_destroy": (None, [vp]),
    "sdr_rrb_reset": (i32, [vp]),
    "sdr_rrb_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_rrb_output_count": (i32, [vp, vp, vp]),
    "sdr_rrb_process": (i32, [vp, vp, vp, sz, vp, sz, sz, vp]),
    "sdr_rrb_process_dev": (i32, [vp, vp, vp, sz, vp, sz, sz, vp]),
    "sdr_arb_step": (i32, [C.c_double, C.c_double, C.POINTER(ArbTime)]),
    "sdr_arb_create": (vp, [C.POINTER(ArbConfig), C.POINTER(i32)]),
    "sdr_arb_destroy": (None, [vp]),
    "sdr_arb_reset": (i32, [vp]),
    "sdr_arb_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_arb_set_steps": (i32, [vp, vp]),
    "sdr_arb_output_count": (i32, [vp, vp, vp]),
    "sdr_arb_process": (i32, [vp, vp, vp, sz, vp, sz, sz, vp]),
    "sdr_arb_process_dev": (i32, [vp, vp, vp, sz, vp, sz, sz, vp]),
    "sdr_tsync_loop_design": (i32, [C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_float),
                                    C.POINTER(C.c_float)]),
    "sdr_tsync_create": (vp, [C.POINTER(TsyncConfig), C.POINTER(i32)]),
    "sdr_tsync_destroy": (None, [vp]),
    "sdr_tsync_reset": (i32, [vp]),
    "sdr_tsync_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_tsync_max_output": (i32, [vp, vp, vp]),
    "sdr_tsync_process": (i32, [vp, vp, vp, sz, vp, vp, vp, sz, sz, vp]),
    "sdr_tsync_process_dev": (i32, [vp, vp, vp, sz, vp, vp, vp, sz, sz, vp]),
    "sdr_tsync_get_state": (i32, [vp, sz, C.POINTER(ArbTime), C.POINTER(C.c_int64)]),
    "sdr_csync_create": (vp, [C.POINTER(CsyncConfig), C.POINTER(i32)]),
    "sdr_csync_destroy": (None, [vp]),
    "sdr_csync_reset": (i32, [vp]),
    "sdr_csync_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_csync_process": (i32, [vp, vp, vp, sz, vp, vp, vp, sz]),
    "sdr_csync_process_dev": (i32, [vp, vp, vp, sz, vp, vp, vp, sz]),
    "sdr_csync_get_state": (i32, [vp, sz, C.POINTER(C.c_uint64), C.POINTER(C.c_int64)]),
    "sdr_eq_create": (vp, [C.POINTER(EqConfig), C.POINTER(i32)]),
    "sdr_eq_destroy": (None, [vp]),
    "sdr_eq_reset": (i32, [vp]),
    "sdr_eq_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_eq_process": (i32, [vp, vp, vp, sz, vp, vp, sz]),
    "sdr_eq_process_dev": (i32, [vp, vp, vp, sz, vp, vp, sz]),
    "sdr_eq_get_taps": (i32, [vp, sz, vp]),
    "sdr_vit_create": (vp, [C.POINTER(VitConfig), C.POINTER(i32)]),
    "sdr_vit_destroy": (None, [vp]),
    "sdr_vit_reset": (i32, [vp]),
    "sdr_vit_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_vit_output_count": (i32, [vp, vp, vp]),
    "sdr_vit_process": (i32, [vp, vp, vp, sz, vp, sz, vp]),
    "sdr_vit_process_dev": (i32, [vp, vp, vp, sz, vp, sz, vp]),
    "sdr_vit_finish": (i32, [vp, vp, i32, vp, sz, vp]),
    "sdr_vit_finish_dev": (i32, [vp, vp, i32, vp, sz, vp]),
    "sdr_fsync_create": (vp, [C.POINTER(FsyncConfig), C.POINTER(i32)]),
    "sdr_fsync_destroy": (None, [vp]),
    "sdr_fsync_reset": (i32, [vp]),
    "sdr_fsync_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_fsync_max_output": (i32, [vp, vp, vp, vp]),
    "sdr_fsync_process": (i32, [vp, vp, vp, sz, vp, sz, sz, vp, vp, sz, sz, vp]),
    "sdr_fsync_process_dev": (i32, [vp, vp, vp, sz, vp, sz, sz, vp, vp, sz, sz, vp]),
    "sdr_fsync_get_state": (i32, [vp, sz, C.POINTER(FsyncState)]),
    "sdr_fm_create": (vp, [C.POINTER(FmConfig), C.POINTER(i32)]),
    "sdr_fm_destroy": (None, [vp]),
    "sdr_fm_reset": (i32, [vp]),
    "sdr_fm_output_rate": (f32, [vp]),
    "sdr_fm_max_output": (sz, [vp, sz]),
    "sdr_fm_process": (i32, [vp, vp, sz, sz, vp, sz, sz, C.POINTER(sz), i32]),
    "sdr_fm_process_dev": (i32, [vp, vp, sz, sz, vp, sz, sz, C.POINTER(sz), i32]),
    "sdr_biquad_create": (vp, [C.POINTER(BiquadConfig), C.POINTER(i32)]),
    "sdr_biquad_destroy": (None, [vp]),
    "sdr_biquad_reset": (i32, [vp]),
    "sdr_biquad_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_biquad_process": (i32, [vp, vp, sz, sz, vp, sz]),
    "sdr_biquad_process_dev": (i32, [vp, vp, sz, sz, vp, sz]),
    "sdr_channelizer_create": (vp, [C.POINTER(FirConfig), C.POINTER(PllConfig), C.POINTER(i32)]),
    "sdr_channelizer_destroy": (None, [vp]),
    "sdr_channelizer_reset": (i32, [vp]),
    "sdr_channelizer_process": (i32, [vp, vp, sz, sz, vp, vp, sz]),
    "sdr_channelizer_process_dev": (i32, [vp, vp, sz, sz, vp, vp, sz]),
    "sdr_src_new": (vp, [i32, i32, C.POINTER(i32)]),
    "sdr_src_new_on": (vp, [i32, i32, i32, vp, C.POINTER(i32)]),
    "sdr_src_delete": (vp, [vp]),
    "sdr_src_process": (i32, [vp, C.POINTER(SrcData)]),
    "sdr_src_process_dev": (i32, [vp, C.POINTER(SrcData)]),
    "sdr_src_reset": (i32, [vp]),
    "sdr_src_clone": (vp, [vp, C.POINTER(i32)]),
    "sdr_src_set_ratio": (i32, [vp, C.c_double]),
    "sdr_src_get_channels": (i32, [vp]),
    "sdr_src_history_frames": (C.c_long, [vp]),
    "sdr_src_set_exact": (i32, [vp, i32]),
    "sdr_src_strerror": (C.c_char_p, [i32]),
    "sdr_src_get_name": (C.c_char_p, [i32]),
    "sdr_src_get_description": (C.c_char_p, [i32]),
    "sdr_src_get_version": (C.c_char_p, []),
    "sdr_src_sinc_table": (sz, [i32, C.POINTER(vp), C.POINTER(i32)]),
    "sdr_timer_create": (vp, [i32, vp, C.POINTER(i32)]),
    "sdr_timer_destroy": (None, [vp]),
    "sdr_timer_begin": (i32, [vp]),
    "sdr_timer_end": (i32, [vp, C.POINTER(f32)]),
    "sdr_kernel_launch_count": (C.c_uint64, []),
}

_lib = None


class SdrError(RuntimeError):
    def __init__(self, code, what=""):
        self.code = code
        msg = lib().sdr_strerror(code)
        super().__init__("%s: [%d] %s" % (what, code, msg.decode() if msg else "?"))


def lib():
    """The loaded C-ABI library.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libsdr_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C unnamed-rust-sdr_b200/csrc`. There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        raise SdrError(rc, what)

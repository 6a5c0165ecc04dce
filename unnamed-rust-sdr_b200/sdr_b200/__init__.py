"""sdr_b200 -- Python view of libsdr_b200.so, the B200 (sm_100a) implementation of the
sample-stream hot path of agrif/unnamed-rust-sdr.  Module layout follows the reference crate
(filter / resample / fft / signal).  There is no CPU fallback: constructing any operator without
the built CUDA library or without a CUDA device raises."""
from . import _ffi
from ._ffi import (FMT_C64, FMT_F32, FMT_U8IQ, LIB_PATH, PROTOTYPES, SdrError, lib)
from .ops import (Arb, Biquad, BiquadD, Channelizer, ConverterType, Csync, Ddc, Duc, Eq, Fcfb, Fcsb, FftPlan, Fir,
                  FmStereo, Fsync, Identity, Pfb, Pfs, PllBatch, PllDesign, Psd, ResampleError, Rrb, SampleRate, Timer, Tsync,
                  Vit, WindowFft, arb_step, block_samples, ddc_phase_increment, decimate_wait, device_count, device_info,
                  duration_samples, fcfb_geometry, fft, fft_labels, kernel_launch_count, rfft, sinc_table,
                  tsync_loop_design, unpack_u8iq, unpack_u8iq_dev)
from . import rtltcp, shard, signal

__all__ = [n for n in dir() if not n.startswith("_")]

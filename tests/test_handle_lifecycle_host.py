"""CPU: the lifecycle contract every handle of the C ABI shares.  A NULL configuration is INVALID_ARG (100) and a NULL
err pointer is accepted; a valid configuration fails with NO_DEVICE (102) on a machine without a GPU; clone and reset
of a NULL handle give NULL_HANDLE (103), BAD_STATE (2) for the libsamplerate-shaped sdr_src; destroy of NULL is a
no-op."""
import ctypes as C

import numpy as np
import pytest


def _keep(keep, a):
    keep.append(a)
    return a.ctypes.data


def _pll_designs(F, keep):
    bq = F.BiquadDesign(F.BQ_LOWPASS, 1000.0, 0.7)
    arr = (F.PllDesign * 1)(F.PllDesign(0.0, 0.01, bq, F.BiquadDesign(F.BQ_IDENTITY, 0.0, 0.0), bq))
    keep.append(arr)
    return C.cast(arr, C.c_void_p)


def _valid(name, F, keep):
    """(create arguments before `err`) of a configuration that is valid on any device"""
    taps = lambda n: _keep(keep, np.ones(n, np.float32))
    u64 = lambda *v: _keep(keep, np.array(v, np.uint64))
    usz = lambda *v: _keep(keep, np.array(v, np.uintp))
    if name == "fir":
        return (C.byref(F.FirConfig(taps(16), 16, 0, F.FMT_C64, 1, 1, 0, 0, None)),)
    if name == "fft":
        return (C.byref(F.FftConfig(1024, F.FMT_C64, 0, 0, None)),)
    if name == "pll":
        return (C.byref(F.PllConfig(_pll_designs(F, keep), 1, 1, 48000.0, 0, 0, None)),)
    if name == "biquad":
        bq = (F.BiquadDesign * 1)(F.BiquadDesign(F.BQ_LOWPASS, 1000.0, 0.7))
        keep.append(bq)
        return (C.byref(F.BiquadConfig(C.cast(bq, C.c_void_p), 1, 1, 48000.0, 0, 0, None)),)
    if name == "src":
        return (F.SRC_SINC_FASTEST, 1, 0, None)
    if name == "pfb":
        return (C.byref(F.PfbConfig(taps(64), 64, 8, 8, F.FMT_C64, 0, 0, None)),)
    if name == "pfs":
        return (C.byref(F.PfsConfig(taps(64), 64, 8, 8, 0, 0, None)),)
    if name == "ddc":
        return (C.byref(F.DdcConfig(taps(32), 32, 1, u64(1 << 60, 3), 2, 4, 0, F.FMT_C64, 0, 0, None)),)
    if name == "duc":
        return (C.byref(F.DucConfig(taps(32), 32, 1, u64(1 << 60, 3), 2, 4, 0, 0, 0, None)),)
    if name == "psd":
        return (C.byref(F.PsdConfig(1024, 512, 4, None, F.FMT_C64, 0, 0, None)),)
    if name == "fcfb":
        return (C.byref(F.FcfbConfig(taps(32), 32, 1, u64(1 << 60, 3), usz(4, 8), 2, 0, F.FMT_C64, 0, None)),)
    if name == "fcsb":
        return (C.byref(F.FcsbConfig(taps(32), 32, 1, u64(1 << 60, 3), usz(4, 8), 2, 0, 0, None)),)
    if name == "rrb":
        return (C.byref(F.RrbConfig(taps(32), 32, 1, usz(3, 2), usz(2, 5), 2, 0, None)),)
    if name == "window_fft":
        return (C.byref(F.WindowFftConfig(1000, 100, F.FMT_C64, 0, 0, None)),)
    if name == "fm":
        return (C.byref(F.FmConfig(1, 1.8e6, 0.0, 0, 0, None)),)
    if name == "channelizer":
        fc = F.FirConfig(taps(16), 16, 0, F.FMT_C64, 1, 2, 0, 0, None)
        pc = F.PllConfig(_pll_designs(F, keep), 1, 2, 48000.0, 0, 0, None)
        keep += [fc, pc]
        return C.byref(fc), C.byref(pc)
    if name == "timer":
        return (0, None)
    raise AssertionError(name)


# name, create symbol, create arguments (before `err`) that are invalid and the code they give, clone, reset, destroy
HANDLES = [
    ("fir", "sdr_fir_create", (None,), 100, True, True, "sdr_fir_destroy"),
    ("fft", "sdr_fft_create", (None,), 100, False, False, "sdr_fft_destroy"),
    ("pll", "sdr_pll_create", (None,), 100, True, True, "sdr_pll_destroy"),
    ("biquad", "sdr_biquad_create", (None,), 100, True, True, "sdr_biquad_destroy"),
    ("src", "sdr_src_new_on", (0, 0, 0, None), 11, True, True, "sdr_src_delete"),  # channels < 1
    ("pfb", "sdr_pfb_create", (None,), 100, True, True, "sdr_pfb_destroy"),
    ("pfs", "sdr_pfs_create", (None,), 100, True, True, "sdr_pfs_destroy"),
    ("ddc", "sdr_ddc_create", (None,), 100, True, True, "sdr_ddc_destroy"),
    ("duc", "sdr_duc_create", (None,), 100, True, True, "sdr_duc_destroy"),
    ("psd", "sdr_psd_create", (None,), 100, True, True, "sdr_psd_destroy"),
    ("fcfb", "sdr_fcfb_create", (None,), 100, True, True, "sdr_fcfb_destroy"),
    ("fcsb", "sdr_fcsb_create", (None,), 100, True, True, "sdr_fcsb_destroy"),
    ("rrb", "sdr_rrb_create", (None,), 100, True, True, "sdr_rrb_destroy"),
    ("window_fft", "sdr_window_fft_create", (None,), 100, False, True, "sdr_window_fft_destroy"),
    ("fm", "sdr_fm_create", (None,), 100, False, True, "sdr_fm_destroy"),
    ("channelizer", "sdr_channelizer_create", (None, None), 100, False, True, "sdr_channelizer_destroy"),
    ("timer", "sdr_timer_create", (-1, None), None, False, False, "sdr_timer_destroy"),
]
IDS = [h[0] for h in HANDLES]


@pytest.mark.parametrize("name,create,bad,bad_code,cloneable,resettable,destroy", HANDLES, ids=IDS)
def test_invalid_create(sdr, name, create, bad, bad_code, cloneable, resettable, destroy):
    fn = getattr(sdr.lib(), create)
    err = C.c_int(-1)
    assert fn(*bad, C.byref(err)) is None
    if bad_code is not None:  # the timer checks its device first: NO_DEVICE or INVALID_ARG
        assert err.value == bad_code
    assert fn(*bad, None) is None


@pytest.mark.parametrize("name,create,bad,bad_code,cloneable,resettable,destroy", HANDLES, ids=IDS)
def test_valid_create_without_device(sdr, name, create, bad, bad_code, cloneable, resettable, destroy):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    keep = []
    args = _valid(name, sdr._ffi, keep)
    fn = getattr(sdr.lib(), create)
    err = C.c_int(-1)
    assert fn(*args, C.byref(err)) is None and err.value == 102
    assert fn(*args, None) is None


@pytest.mark.parametrize("name,create,bad,bad_code,cloneable,resettable,destroy", HANDLES, ids=IDS)
def test_null_handle(sdr, name, create, bad, bad_code, cloneable, resettable, destroy):
    lib = sdr.lib()
    null_code = 2 if name == "src" else 103
    if cloneable:
        clone = getattr(lib, "sdr_%s_clone" % name)
        err = C.c_int(-1)
        assert clone(None, C.byref(err)) is None and err.value == null_code
        assert clone(None, None) is None
    if resettable:
        assert getattr(lib, "sdr_%s_reset" % name)(None) == null_code
    getattr(lib, destroy)(None)

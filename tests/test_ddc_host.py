"""CPU: the down-converter bank's definition (mix with a 64-bit NCO, filter, decimate) equals the rotated-taps form the
kernels compute; sdr_ddc_phase_increment's rounding; argument validation of sdr_ddc_create; no device means a loud
failure."""
import ctypes as C

import numpy as np
import pytest

import ddc_ref as R
import gen

TWO64 = 1 << 64


@pytest.mark.parametrize("first", [0, 12345, (1 << 63) - 7, TWO64 - 100])
@pytest.mark.parametrize("D", [1, 3, 8])
def test_rotated_taps_form_equals_mix_first(first, D):
    incs = [R.phase_increment_exact(f, 2.4e6) for f in (312.5e3, -687e3, 1.2e6, 0.0, 2.4e6 - 1.0)]
    incs.append((1 << 64) - 1)  # one step below a full turn: wraps every sample
    h = np.stack([gen.lowpass_taps(37, 0.05 + 0.01 * k, 1.0) for k in range(len(incs))]).astype(np.float64)
    x = gen.complex_noise(600, 3 + D).astype(np.complex128)
    want = R.mix_first_f64(h, x, incs, D, first)
    got = R.rotated_f64(h, x, incs, D, first)
    assert got.shape == want.shape == (len(incs), 600 // D)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_definition_matches_oracle_composition():
    """the f64 definition is the crate's blocks (mix in f32, Fir(h), decimate) up to f32 rounding"""
    incs = [R.phase_increment_exact(f, 1.0) for f in (0.13, -0.31)]
    h = gen.lowpass_taps(41, 0.05, 1.0)
    x = gen.complex_noise(700, 9)
    want = R.mix_first_f64(h.astype(np.float64), x, incs, 4)
    got = R.oracle_f32(h, x, incs, 4)
    assert got.shape == want.shape
    for k in range(len(incs)):
        assert np.abs(got[k] - want[k]).max() <= 1e-5 * np.abs(want[k]).max()


@pytest.mark.parametrize("freq,rate,want", [(0.25, 1.0, 1 << 62), (-0.25, 1.0, TWO64 - (1 << 62)), (0.5, 1.0, 1 << 63),
                                            (-0.5, 1.0, 1 << 63), (1.25, 1.0, 1 << 62), (0.0, 1.0, 0),
                                            (2.5, 1.0, 1 << 63), (-1.75, 1.0, 1 << 62)])
def test_phase_increment_known_values(sdr, freq, rate, want):
    assert sdr.ddc_phase_increment(freq, rate) == want
    assert R.phase_increment_exact(freq, rate) == want


@pytest.mark.parametrize("freq,rate", [(100e3, 2.4e6), (-100e3, 2.4e6), (312.5e3, 2.4e6), (-687e3, 2.4e6),
                                       (1.0, 3.0), (2.0, 3.0), (-1e-9, 1.0), (1e-20, 1.0), (123456.789, 2.048e6),
                                       (7.3e6, 2.4e6), (0.49999999999999994, 1.0)])
def test_phase_increment_against_exact_arithmetic(sdr, freq, rate):
    got = sdr.ddc_phase_increment(freq, rate)
    assert got == R.phase_increment_exact(freq, rate)
    # centred where asked: the signed increment over 2^64 is freq / rate folded into [-1/2, 1/2]
    nu = freq / rate - round(freq / rate)
    signed = got - TWO64 if got >= 1 << 63 else got
    assert abs(signed / TWO64 - nu) <= 2.0 ** -64 + 1e-16 * abs(nu)


def test_phase_increment_non_finite_is_zero(sdr):
    assert sdr.ddc_phase_increment(float("nan"), 1.0) == 0
    assert sdr.ddc_phase_increment(1.0, 0.0) == 0
    assert sdr.ddc_phase_increment(float("inf"), 1.0) == 0


def _cfg(sdr, taps, n_taps, n_sets, inc, C_, D, fmt, flags=0):
    return sdr._ffi.DdcConfig(taps.ctypes.data if taps is not None else None, n_taps, n_sets,
                              inc.ctypes.data if inc is not None else None, C_, D, 0, fmt, flags, 0, None)


def test_ddc_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    inc = np.arange(4, dtype=np.uint64)
    many = np.zeros(257, np.uint64)
    assert L.sdr_ddc_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, inc, 4, 8, sdr.FMT_U8IQ),        # NULL taps
           _cfg(sdr, h, 64, 1, None, 4, 8, sdr.FMT_U8IQ),          # NULL increments
           _cfg(sdr, h, 0, 1, inc, 4, 8, sdr.FMT_U8IQ),            # L = 0
           _cfg(sdr, h, 64, 1, inc, 0, 8, sdr.FMT_U8IQ),           # C = 0
           _cfg(sdr, h, 64, 1, many, 257, 8, sdr.FMT_U8IQ),        # beyond the channel limit
           _cfg(sdr, h, 64, 1, inc, 4, 0, sdr.FMT_U8IQ),           # D = 0
           _cfg(sdr, h, 64, 2, inc, 4, 8, sdr.FMT_U8IQ),           # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 0, inc, 4, 8, sdr.FMT_U8IQ),
           _cfg(sdr, h, 64, 1, inc, 4, 8, sdr.FMT_F32),            # real input
           _cfg(sdr, h, 64, 1, inc, 4, 8, 7),
           _cfg(sdr, h, 64, 1, inc, 4, 8, sdr.FMT_U8IQ, 2)]        # unknown flag
    for cfg in bad:
        err.value = 0
        assert L.sdr_ddc_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    nan = h.copy()
    nan[5] = np.nan
    err.value = 0
    assert L.sdr_ddc_create(C.byref(_cfg(sdr, nan, 64, 1, inc, 4, 8, sdr.FMT_U8IQ)), C.byref(err)) is None
    assert err.value == 100
    n = C.c_size_t(7)
    assert L.sdr_ddc_process(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_ddc_process_dev(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_ddc_reset(None) == 103
    assert L.sdr_ddc_output_count(None, 100) == 0
    assert L.sdr_ddc_last_path(None) == 0
    assert L.sdr_ddc_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_ddc_destroy(None)


def test_ddc_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Ddc(gen.lowpass_taps(64, 0.05, 1.0), [100e3, -200e3], 2.4e6, 8)
    assert e.value.code == 102

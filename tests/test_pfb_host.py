"""CPU: the polyphase filter bank's definition (M modulated FIRs + decimate, the crate's blocks) equals the polyphase
form the kernels compute; argument validation of sdr_pfb_create; no device means a loud failure."""
import ctypes as C

import numpy as np
import pytest

import gen
import pfb_ref as R


@pytest.mark.parametrize("M", [4, 8, 16])
@pytest.mark.parametrize("Dsel", ["M", "M/2", 3, 1])
@pytest.mark.parametrize("extra", [0, 3])
def test_polyphase_form_equals_definition(M, Dsel, extra):
    D = {"M": M, "M/2": M // 2}.get(Dsel, Dsel)
    L = 5 * M + extra if extra else 4 * M - 1  # ragged L: partial last branch row, or T*M - 1
    h = gen.lowpass_taps(L, 1.0 / (2 * M), 1.0).astype(np.float64)
    x = gen.complex_noise(40 * M + 7, 11 + M).astype(np.complex128)
    want = R.direct_f64(h, x, M, D)
    got = R.polyphase_f64(h, x, M, D)
    assert got.shape == want.shape == (x.size // D, M)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_direct_definition_matches_oracle_blocks():
    """the f64 definition is the crate's Fir(g_k) + Decimate (through the CPU oracle) up to f32 rounding"""
    M, D = 8, 3
    h = gen.lowpass_taps(37, 1.0 / 16, 1.0)
    x = gen.complex_noise(500, 5)
    want = R.direct_f64(h.astype(np.float64), x, M, D)
    got = R.direct_oracle_f32(h, x, M, D)
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()


def _cfg(sdr, taps, n_taps, M, D, fmt, flags=0):
    return sdr._ffi.PfbConfig(taps.ctypes.data if taps is not None else None, n_taps, M, D, fmt, flags, 0, None)


def test_pfb_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    h = np.ones(64, np.float32)
    assert L.sdr_pfb_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 8, 8, sdr.FMT_C64),          # NULL taps
           _cfg(sdr, h, 0, 8, 8, sdr.FMT_C64),             # L = 0
           _cfg(sdr, h, 64, 1, 1, sdr.FMT_C64),            # M < 2
           _cfg(sdr, h, 64, 0, 1, sdr.FMT_C64),
           _cfg(sdr, h, 64, 8, 0, sdr.FMT_C64),            # D = 0
           _cfg(sdr, h, 64, 8, 8, sdr.FMT_F32),            # real input
           _cfg(sdr, h, 64, 8, 8, 7),
           _cfg(sdr, h, 64, 8, 8, sdr.FMT_C64, 8),         # unknown flag
           _cfg(sdr, h, 64, 1 << 17, 8, sdr.FMT_C64)]      # beyond the channel limit
    for cfg in bad:
        err.value = 0
        assert L.sdr_pfb_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    n = C.c_size_t(7)
    assert L.sdr_pfb_process(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_pfb_process_dev(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_pfb_reset(None) == 103
    assert L.sdr_pfb_output_count(None, 100) == 0
    assert L.sdr_pfb_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_pfb_destroy(None)


def test_pfb_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Pfb(gen.lowpass_taps(64, 0.5 / 8, 1.0), 8, 8, "u8iq")
    assert e.value.code == 102

"""CPU: the fast-convolution bank's overlap-save computation (absolute block grid, spectral fold by the power-of-two part
of D_k, pick, derotation) equals the definition (sdr_ddc's channel with its own D_k); sdr_fcfb_geometry equals the
documented rule; output counts; argument validation of sdr_fcfb_create; no device means a loud failure."""
import ctypes as C

import numpy as np
import pytest

import ddc_ref as R
import fcfb_ref as Q
import gen


def _incs(C_, seed):
    rng = np.random.default_rng(seed)
    incs = [R.phase_increment_exact(f, 1.0) for f in rng.uniform(-0.5, 0.5, C_)]
    incs[0] = (1 << 64) - 1  # one step below a full turn: wraps every sample
    return incs


@pytest.mark.parametrize("first", [0, 12345, 7, (1 << 40) + 12345, (1 << 63) - 7])
@pytest.mark.parametrize("ds", [[1, 2, 8, 10, 40], [10], [8, 8, 16, 32], [3, 5]])
def test_overlap_save_equals_definition(first, ds):
    rng = np.random.default_rng(len(ds) + first % 97)
    L = int(rng.integers(1, 700))
    h = np.stack([gen.lowpass_taps(L, 0.05 + 0.01 * k, 1.0) if L > 1 else np.array([0.5 + 0.1 * k], np.float32)
                  for k in range(len(ds))]).astype(np.float64)
    incs = _incs(len(ds), L)
    N, P = Q.geometry(L, ds)
    n = 3 * N + int(rng.integers(0, N))
    x = gen.complex_noise(n, 3 + L).astype(np.complex128)
    want = Q.definition_f64(h, x, incs, ds, first)
    got = Q.overlap_save_f64(h, x, incs, ds, first)
    o0 = Q.off0(first, ds, P)
    for k, d in enumerate(ds):
        assert got[k].size == Q.counts(n, ds, P, o0)[k]
        assert n // d - P // d <= got[k].size <= n // d  # released at most P - 1 samples late
        assert np.abs(got[k] - want[k][:got[k].size]).max() <= 1e-12 * np.abs(want[k]).max()


def test_overlap_save_shared_taps_equal_ddc_definition():
    """every D_k = D: the same function as sdr_ddc"""
    h = gen.lowpass_taps(255, 0.04, 1.0).astype(np.float64)
    incs = _incs(3, 5)
    x = gen.complex_noise(5000, 4).astype(np.complex128)
    got = Q.overlap_save_f64(h, x, incs, [8, 8, 8], 999)
    want = R.mix_first_f64(h, x, incs, 8, 999)
    for k in range(3):
        assert np.abs(got[k] - want[k][:got[k].size]).max() <= 1e-12 * np.abs(want[k]).max()


GEOMETRY_CASES = [(1, [1]), (64, [1]), (255, [8]), (511, [10]), (512, [1, 2, 8, 10, 40]), (4095, [8] * 8),
                  (4095, [8, 8, 16, 16, 32, 32, 64, 64]), (65537, [1]), (1 << 20, [1]), (1 << 20, [3]), (100, [1000]),
                  (100, [4096]), (1, [1 << 22]), (1, [(1 << 22) + 1]), (10, [2 ** 11, 3 ** 7]), (1 << 20, [1 << 21])]


@pytest.mark.parametrize("L,ds", GEOMETRY_CASES)
def test_geometry_matches_rule(sdr, L, ds):
    d = np.array(ds, np.uintp)
    n, p = C.c_size_t(0), C.c_size_t(0)
    rc = sdr.lib().sdr_fcfb_geometry(L, d.ctypes.data, d.size, C.byref(n), C.byref(p))
    want = Q.geometry(L, ds)
    if want is None:
        assert rc == 101
        return
    assert rc == 0 and (n.value, p.value) == want
    N, P = want
    assert N & (N - 1) == 0 and 1024 <= N <= 1 << 22
    assert N - P >= L - 1 and P % Q.lcm_of(ds) == 0 and 2 * P >= N
    assert sdr.fcfb_geometry(L, ds) == want


def test_counts_across_call_sequences():
    ds = [1, 2, 8, 10, 40]
    N, P = Q.geometry(300, ds)
    for first in (0, 40 * 7 + 3, (1 << 63) - 7):
        o0 = Q.off0(first, ds, P)
        assert o0 % Q.lcm_of(ds) == 0 and 0 <= o0 < P
        rng = np.random.default_rng(first % 1000)
        total, got = 0, [0] * len(ds)
        for step in list(rng.integers(0, 3 * P, 40)) + [1] * 50 + [P - 1, 1, 0]:
            before = Q.counts(total, ds, P, o0)
            total += int(step)
            after = Q.counts(total, ds, P, o0)
            got = [g + a - b for g, a, b in zip(got, after, before)]
        assert got == Q.counts(total, ds, P, o0)
        for k, d in enumerate(ds):
            assert total // d - P // d <= got[k] <= total // d


def _cfg(sdr, taps, n_taps, n_sets, inc, dec, C_, fmt):
    return sdr._ffi.FcfbConfig(taps.ctypes.data if taps is not None else None, n_taps, n_sets,
                               inc.ctypes.data if inc is not None else None,
                               dec.ctypes.data if dec is not None else None, C_, 0, fmt, 0, None)


def test_fcfb_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    inc = np.arange(4, dtype=np.uint64)
    dec = np.array([1, 2, 8, 10], np.uintp)
    zero = np.array([1, 0, 8, 10], np.uintp)
    many = np.zeros(257, np.uint64)
    many_d = np.ones(257, np.uintp)
    assert L.sdr_fcfb_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, inc, dec, 4, sdr.FMT_U8IQ),        # NULL taps
           _cfg(sdr, h, 64, 1, None, dec, 4, sdr.FMT_U8IQ),          # NULL increments
           _cfg(sdr, h, 64, 1, inc, None, 4, sdr.FMT_U8IQ),          # NULL decimations
           _cfg(sdr, h, 0, 1, inc, dec, 4, sdr.FMT_U8IQ),            # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, inc, dec, 4, sdr.FMT_U8IQ),  # L beyond 2^20
           _cfg(sdr, h, 64, 1, inc, dec, 0, sdr.FMT_U8IQ),           # C = 0
           _cfg(sdr, h, 64, 1, many, many_d, 257, sdr.FMT_U8IQ),     # beyond the channel limit
           _cfg(sdr, h, 64, 1, inc, zero, 4, sdr.FMT_U8IQ),          # D_k = 0
           _cfg(sdr, h, 64, 2, inc, dec, 4, sdr.FMT_U8IQ),           # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 0, inc, dec, 4, sdr.FMT_U8IQ),
           _cfg(sdr, h, 64, 1, inc, dec, 4, sdr.FMT_F32),            # real input
           _cfg(sdr, h, 64, 1, inc, dec, 4, 7)]
    for cfg in bad:
        err.value = 0
        assert L.sdr_fcfb_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    nan = h.copy()
    nan[5] = np.nan
    err.value = 0
    assert L.sdr_fcfb_create(C.byref(_cfg(sdr, nan, 64, 1, inc, dec, 4, sdr.FMT_U8IQ)), C.byref(err)) is None
    assert err.value == 100
    huge = np.array([(1 << 22) + 1], np.uintp)                     # no N <= 2^22 fits
    err.value = 0
    assert L.sdr_fcfb_create(C.byref(_cfg(sdr, h, 64, 1, inc, huge, 1, sdr.FMT_U8IQ)), C.byref(err)) is None
    assert err.value == 101
    n, p = C.c_size_t(0), C.c_size_t(0)
    assert L.sdr_fcfb_geometry(64, None, 1, C.byref(n), C.byref(p)) == 100
    assert L.sdr_fcfb_geometry(0, dec.ctypes.data, 4, C.byref(n), C.byref(p)) == 100
    assert L.sdr_fcfb_geometry(64, zero.ctypes.data, 4, C.byref(n), C.byref(p)) == 100
    assert L.sdr_fcfb_geometry(64, dec.ctypes.data, 0, C.byref(n), C.byref(p)) == 100
    assert L.sdr_fcfb_geometry(64, dec.ctypes.data, 4, None, C.byref(p)) == 100
    cnt = np.zeros(4, np.uintp)
    assert L.sdr_fcfb_process(None, None, 0, None, 0, 0, cnt.ctypes.data) == 103
    assert L.sdr_fcfb_process_dev(None, None, 0, None, 0, 0, cnt.ctypes.data) == 103
    assert L.sdr_fcfb_output_count(None, 100, cnt.ctypes.data) == 103
    assert L.sdr_fcfb_reset(None) == 103
    assert L.sdr_fcfb_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_fcfb_destroy(None)


def test_fcfb_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Fcfb(gen.lowpass_taps(64, 0.05, 1.0), [100e3, -200e3], 2.4e6, [8, 10])
    assert e.value.code == 102

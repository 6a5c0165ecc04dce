"""CPU: the power-spectrum estimator's f64 reference equals a literal restatement of the crate chain; the library's
chunked summation order is the plain mean; output_count arithmetic; argument validation of sdr_psd_create; no device
means a loud failure."""
import ctypes as C

import numpy as np
import pytest

import gen
import psd_ref as R


@pytest.mark.parametrize("N,H,K", [(16, 16, 1), (16, 8, 3), (16, 4, 2), (16, 3, 5), (16, 33, 2), (12, 5, 4), (1, 1, 3),
                                   (7, 2, 1)])
@pytest.mark.parametrize("taper", [False, True])
@pytest.mark.parametrize("shift,norm", [(True, True), (False, False), (True, False)])
def test_reference_equals_literal_chain(N, H, K, taper, shift, norm):
    x = gen.complex_noise(300, 11 + N + H).astype(np.complex128)
    w = np.hanning(N) if taper else None
    want = R.power_literal(x, N, H, K, w, shift, norm)
    got = R.power_f64(x, N, H, K, w, shift, norm)
    assert got.shape == want.shape and got.shape[0] == R.spectra_count(300, H, K) > 0
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("K", [1, 5, 32, 33, 64, 100])
def test_chunked_order_equals_plain_mean(K):
    rng = np.random.default_rng(K)
    p = rng.random((3 * K, 24)).astype(np.float32).astype(np.float64)
    got = R.chunked(p, K)
    want = p.reshape(3, K, 24).mean(axis=1)
    # f32 chunk sums of <= 32 terms: the only rounding beyond f64
    assert np.abs(got - want).max() <= 32 * 2.0 ** -24 * want.max()


def _count_model(calls, H, K):
    total, out = 0, []
    for n in calls:
        out.append(((total + n) // H) // K - (total // H) // K)
        total += n
    return out


@pytest.mark.parametrize("H,K", [(1, 1), (3, 1), (1024, 256), (512, 33), (1041, 5)])
def test_output_count_on_ragged_calls(H, K):
    rng = np.random.default_rng(H + K)
    calls = [int(v) for v in rng.integers(0, 5 * H * K, 40)] + [0, 1, 1, H * K - 1, 1]
    counts = _count_model(calls, H, K)
    assert sum(counts) == R.spectra_count(sum(calls), H, K)
    assert all(c >= 0 for c in counts)


def _cfg(sdr, n, hop, avg, fmt, window=None, flags=0):
    return sdr._ffi.PsdConfig(n, hop, avg, window.ctypes.data if window is not None else None, fmt, flags, 0, None)


def test_psd_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    assert L.sdr_psd_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, 0, 1024, 1, sdr.FMT_U8IQ),         # N = 0
           _cfg(sdr, 1024, 0, 1, sdr.FMT_U8IQ),         # H = 0
           _cfg(sdr, 1024, 1024, 0, sdr.FMT_U8IQ),      # K = 0
           _cfg(sdr, 1024, 1024, 1, sdr.FMT_F32),       # real input
           _cfg(sdr, 1024, 1024, 1, 7),
           _cfg(sdr, 1024, 1024, 1, sdr.FMT_C64, flags=8)]  # unknown flag
    for cfg in bad:
        err.value = 0
        assert L.sdr_psd_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    n = C.c_size_t(7)
    assert L.sdr_psd_process(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_psd_process_dev(None, None, 0, None, 0, 0, C.byref(n)) == 103
    assert L.sdr_psd_reset(None) == 103
    assert L.sdr_psd_output_count(None, 100) == 0
    assert L.sdr_psd_last_path(None) == 0
    assert L.sdr_psd_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_psd_destroy(None)


def test_psd_python_rejects_wrong_window_length(sdr):
    with pytest.raises(ValueError):
        sdr.Psd(1024, 1024, 4, window=np.ones(1000, np.float32))


def test_psd_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Psd(1024, 512, 8, window=np.hanning(1024))
    assert e.value.code == 102

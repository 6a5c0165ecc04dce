"""CPU: the synthesis bank's definition (zero-stuff + M modulated FIRs + sum, the crate's blocks) equals the polyphase
form the kernels compute; the analysis -> synthesis round trip with the Kaiser prototype pair; output counts, argument
validation of sdr_pfs_create and the loud failure without a device."""
import ctypes as C

import numpy as np
import pytest

import gen
import pfb_ref
import pfs_ref as R


def _frames(n, M, seed):
    return gen.complex_noise(n * M, seed).reshape(n, M)


@pytest.mark.parametrize("M", [4, 8, 16])
@pytest.mark.parametrize("Dsel", ["M", "M/2", 3, 1])
@pytest.mark.parametrize("L", ["ragged", "T*M-1", 1])
def test_polyphase_form_equals_definition(M, Dsel, L):
    D = {"M": M, "M/2": M // 2}.get(Dsel, Dsel)
    L = {"ragged": 5 * M + 3, "T*M-1": 4 * M - 1}.get(L, L)  # not a multiple of M (nor of D unless D = 1)
    f = gen.lowpass_taps(L, 1.0 / M, 1.0).astype(np.float64) if L > 1 else np.array([0.75])
    y = _frames(40, M, 11 + M + D).astype(np.complex128)
    want = R.direct_f64(f, y, M, D)
    got = R.polyphase_f64(f, y, M, D)
    assert got.shape == want.shape == (40 * D,)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    # a subset of outputs is the same as the whole
    pick = np.array([0, 1, D - 1, 17 * D + 2, 40 * D - 1])
    assert np.abs(R.polyphase_f64(f, y, M, D, outputs=pick) - want[pick]).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("M,D", [(8, 8), (8, 3), (16, 8)])
def test_definition_matches_oracle_blocks(M, D):
    """the f64 definition is zero-stuff + the crate's Fir(f_k) + sum (through the CPU oracle) within the FFT bar"""
    f = gen.lowpass_taps(5 * M + 3, 1.0 / M, 1.0)
    y = _frames(60, M, 5)
    want = R.direct_f64(f.astype(np.float64), y, M, D)
    got = R.direct_oracle_f32(f, y, M, D)
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-5 * np.log2(M) * np.abs(want).max()


@pytest.mark.parametrize("M,D,T", [(16, 8, 12), (64, 32, 12)])
def test_round_trip_reconstructs_the_input_f64(M, D, T):
    """pfb polyphase (h) -> pfs polyphase (f): x[t - T M] with unit gain and >= 100 dB SNR once the gain is fitted"""
    h, f = R.prototype_pair(M, D, T)
    n = 400 * M
    x = gen.complex_noise(n, 3).astype(np.complex128)
    y = pfb_ref.polyphase_f64(h, x, M, D)
    xr = R.polyphase_f64(f, y, M, D)
    assert xr.size == n
    d = T * M
    a, b = 2 * d, n
    ref = x[a - d:b - d]
    gain = np.vdot(ref, xr[a:b]) / np.vdot(ref, ref)
    snr = 10 * np.log10(np.mean(np.abs(gain * ref) ** 2) / np.mean(np.abs(xr[a:b] - gain * ref) ** 2))
    assert abs(gain - 1) < 1e-4
    assert snr >= 100, snr


def _cfg(sdr, taps, n_taps, M, D, flags=0):
    return sdr._ffi.PfsConfig(taps.ctypes.data if taps is not None else None, n_taps, M, D, flags, 0, None)


def test_pfs_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    f = np.ones(64, np.float32)
    assert L.sdr_pfs_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 8, 8),          # NULL taps
           _cfg(sdr, f, 0, 8, 8),             # L = 0
           _cfg(sdr, f, 64, 1, 1),            # M < 2
           _cfg(sdr, f, 64, 0, 1),
           _cfg(sdr, f, 64, 8, 0),            # D = 0
           _cfg(sdr, f, 64, 8, 8, 8),         # unknown flag
           _cfg(sdr, f, 64, 1 << 17, 8)]      # beyond the channel limit
    for cfg in bad:
        err.value = 0
        assert L.sdr_pfs_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    n = C.c_size_t(7)
    assert L.sdr_pfs_process(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert L.sdr_pfs_process_dev(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert L.sdr_pfs_reset(None) == 103
    assert L.sdr_pfs_output_count(None, 100) == 0
    assert L.sdr_pfs_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_pfs_destroy(None)


def test_pfs_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Pfs(gen.lowpass_taps(64, 1.0 / 8, 1.0), 8, 4)
    assert e.value.code == 102


@pytest.mark.parametrize("L,D", [(1, 1), (2, 1), (12 * 1024 + 1, 512), (12 * 1024 + 1, 1024), (100, 7), (7, 100)])
def test_carried_frames_and_drain_count(L, D):
    """frame m releases outputs [m D, (m+1) D); the oldest frame they reach is m - ceil((L - 1) / D), the number of
    frames the handle carries, and as many zero frames flush the tail of the last real frame"""
    H = -(-(L - 1) // D)
    m = 5
    reach = 0
    for t in range(m * D, (m + 1) * D):
        c = (t + 1) % D
        if c < L:
            n_max = c + (L - 1 - c) // D * D  # the last tap of output t
            reach = max(reach, m - ((t + 1 - n_max) // D - 1))
    assert reach == H
    last = D - 1 + L - 1  # the last output frame 0 reaches
    assert last // D == H

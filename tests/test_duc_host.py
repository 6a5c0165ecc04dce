"""CPU: the up-converter bank's computed form equals its definition (zero-stuff, np.convolve, exact integer-phase mixer,
sum); the adjoint identity that pins it against sdr_ddc; the f64 ddc -> duc round trip with a Kaiser pair; output
counts, argument validation of sdr_duc_create and the loud failure without a device."""
import ctypes as C

import numpy as np
import pytest

import ddc_ref
import duc_ref as R
import gen

F_BIG = (1 << 40) + 12345
F_TOP = (1 << 63) - 7
ROUND_TRIP_SNR_DB = 106.0  # the f64 figure of the D = 8, T = 64, beta = 10 pair below (106.4 dB)


def _incs(C_, seed):
    rng = np.random.default_rng(seed)
    return [ddc_ref.phase_increment_exact(float(f), 1.0) for f in rng.uniform(-0.5, 0.5, C_)]


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n).astype(np.complex128)


def _taps(C_, L, shared, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(L if shared else (C_, L))


@pytest.mark.parametrize("C_", [1, 3, 17])
@pytest.mark.parametrize("I", [1, 3, 8])
@pytest.mark.parametrize("L", [1, 2, 64, 255])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("F", [0, F_BIG, F_TOP])
def test_computed_form_equals_definition(C_, I, L, shared, F):
    h = _taps(C_, L, shared, L + C_)
    y = _rows(C_, 40, 3 + I)
    incs = _incs(C_, C_ + I)
    want = R.definition_f64(h, y, incs, I, F)
    got = R.computed_f64(h, y, incs, I, F)
    assert got.shape == want.shape == (40 * I,)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    pick = np.array([0, I - 1, 17 * I + 1, 40 * I - 1])
    assert np.abs(R.computed_f64(h, y, incs, I, F, outputs=pick) - want[pick]).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("C_,D,L,F", [(3, 5, 23, F_BIG), (1, 1, 7, 0), (4, 8, 64, F_TOP), (2, 3, 1, 5)])
def test_adjoint_of_ddc(C_, D, L, F):
    """<v, ddc(x)> = <duc'(v), x> with duc' = (I = D, reversed taps, first_sample F - (L - 1), v followed by
    ceil((L - 1) / D) zero frames) and x-hat read from sample L - 1 on"""
    rng = np.random.default_rng(C_ + D + L)
    incs = _incs(C_, D)
    h = rng.standard_normal((C_, L))
    nf = 37
    x = rng.standard_normal(nf * D) + 1j * rng.standard_normal(nf * D)
    v = rng.standard_normal((C_, nf)) + 1j * rng.standard_normal((C_, nf))
    H = -(-(L - 1) // D)
    xh = R.computed_f64(h[:, ::-1], np.concatenate([v, np.zeros((C_, H))], axis=1), incs, D,
                        (F - (L - 1)) % (1 << 64))
    lhs = np.sum(np.conj(v) * ddc_ref.mix_first_f64(h, x, incs, D, F))
    rhs = np.sum(np.conj(xh[L - 1:L - 1 + nf * D]) * x)
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs)


def round_trip_input(n, F, nus, bw=0.02, seed=10):
    """C band-limited components (|f| < bw), component k mixed up to nus[k] by the exact NCO at absolute index F + n"""
    incs = [ddc_ref.phase_increment_exact(nu, 1.0) for nu in nus]
    x = np.zeros(n, np.complex128)
    for k, inc in enumerate(incs):
        x += R.band_limited(n, bw, seed + k) * R.rot_up(ddc_ref.phases(F, np.arange(n), inc))
    return x, incs


def test_round_trip_reconstructs_the_input_f64():
    """ddc(h) -> duc(f = D h, first_sample F - d): x[n - d] with d = T D, channels at -0.3, 0.05, 0.27 of the rate"""
    D, T = 8, 64
    h, f = R.kaiser_pair(D, T)
    n, F = 1 << 15, F_BIG
    x, incs = round_trip_input(n, F, (-0.3, 0.05, 0.27))
    y = ddc_ref.mix_first_f64(h, x, incs, D, F)
    d = T * D
    xr = R.computed_f64(f, y, incs, D, (F - d) % (1 << 64))
    assert xr.size == n
    ref = x[3 * d:n - d]
    snr = 10 * np.log10(np.mean(np.abs(ref) ** 2) / np.mean(np.abs(xr[4 * d:] - ref) ** 2))
    assert snr >= ROUND_TRIP_SNR_DB, snr
    # without the delay correction channel k comes back rotated by e^{+2 pi i d Delta_k / 2^64}
    xw = R.computed_f64(f, y, incs, D, F)
    assert np.mean(np.abs(xw[4 * d:] - ref) ** 2) > 0.1 * np.mean(np.abs(ref) ** 2)


@pytest.mark.parametrize("L,I", [(1, 1), (2, 1), (255, 8), (4095, 8), (100, 7), (7, 100)])
def test_carried_frames_and_drain_count(L, I):
    """frame m releases outputs [m I, (m+1) I); frame m's last nonzero output is (m+1) I - 1 + L - 1, inside the
    outputs of the H = ceil((L - 1) / I) frames after it"""
    H = -(-(L - 1) // I)
    m = 5
    last = (m + 1) * I - 1 + L - 1
    assert last // I == m + H


def _cfg(sdr, taps, L, sets, incs, C_, I, flags=0, first=0):
    return sdr._ffi.DucConfig(None if taps is None else taps.ctypes.data, L, sets,
                              None if incs is None else incs.ctypes.data, C_, I, first, flags, 0, None)


def test_duc_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    inc = np.zeros(300, np.uint64)
    assert lib.sdr_duc_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, inc, 4, 8),          # NULL taps
           _cfg(sdr, h, 64, 1, None, 4, 8),            # NULL increments
           _cfg(sdr, h, 0, 1, inc, 4, 8),              # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, inc, 4, 8),  # L > 2^20
           _cfg(sdr, h, 64, 1, inc, 0, 8),             # C = 0
           _cfg(sdr, h, 64, 1, inc, 257, 8),           # C > 256
           _cfg(sdr, h, 64, 2, inc, 4, 8),             # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 1, inc, 4, 0),             # I = 0
           _cfg(sdr, h, 64, 1, inc, 4, 8, flags=1)]    # unknown flag
    for cfg in bad:
        err.value = 0
        assert lib.sdr_duc_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    n = C.c_size_t(7)
    assert lib.sdr_duc_process(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert lib.sdr_duc_process_dev(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert lib.sdr_duc_reset(None) == 103
    assert lib.sdr_duc_output_count(None, 100) == 0
    assert lib.sdr_duc_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_duc_destroy(None)


def test_duc_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Duc(gen.lowpass_taps(64, 1.0 / 8, 1.0), [0.1, -0.2], 1.0, 8)
    assert e.value.code == 102

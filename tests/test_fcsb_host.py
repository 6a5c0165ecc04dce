"""CPU: the fast-convolution synthesis bank's overlap-save form (rotated frames, unfold by the power-of-two part of I_k,
sum over channels, one N-point inverse) equals its definition (zero-stuff, np.convolve, exact integer-phase mixer,
sum); with every I_k equal the definition is sdr_duc's; the adjoint identity that pins it against sdr_fcfb; the f64
fcfb -> fcsb round trip at mixed rates; output counts and draining; argument validation of sdr_fcsb_create; no device
means a loud failure."""
import ctypes as C

import numpy as np
import pytest

import ddc_ref as R
import duc_ref
import fcfb_ref
import fcsb_ref as Q
import gen

F_BIG = (1 << 40) + 12345
F_TOP = (1 << 63) - 7
TWO64 = 1 << 64
ROUND_TRIP_SNR_DB = 100.0


def _incs(C_, seed):
    rng = np.random.default_rng(seed)
    incs = [R.phase_increment_exact(float(f), 1.0) for f in rng.uniform(-0.5, 0.5, C_)]
    incs[0] = (1 << 64) - 1  # one step below a full turn: wraps every sample
    return incs


def _rows(Is, n_time, seed):
    return [gen.complex_noise(n_time // int(I), seed + k).astype(np.complex128) for k, I in enumerate(Is)]


def _taps(C_, L, seed):
    return np.random.default_rng(seed).standard_normal((C_, L))


@pytest.mark.parametrize("first", [0, F_BIG, F_TOP])
@pytest.mark.parametrize("L", [1, 2, 255, 1024, 4095])
@pytest.mark.parametrize("Is", [[8], [8, 10, 1, 40, 2], [3, 5, 7], [1]])
def test_overlap_save_equals_definition(Is, L, first):
    h = _taps(len(Is), L, L + len(Is))
    incs = _incs(len(Is), L)
    N, P = Q.geometry(L, Is)
    Il = Q.lcm_of(Is)
    n = -(-(2 * N + 777) // Il) * Il
    rows = _rows(Is, n, 3 + L)
    want = Q.definition_f64(h, rows, incs, Is, first)
    got = Q.overlap_save_f64(h, rows, incs, Is, first)
    o0 = Q.off0(first, Is, P)
    assert o0 % Il == 0 and 0 <= o0 < P
    assert got.size == Q.counts(n, P, o0)
    assert n - P < got.size <= n  # released at most P - Il positions late
    assert np.abs(got - want[:got.size]).max() <= 1e-12 * np.abs(want).max()


def test_equal_interpolations_are_duc():
    """every I_k = I: the definition is sdr_duc's"""
    I, L = 8, 255
    h = _taps(3, L, 1)
    incs = _incs(3, 5)
    y = np.stack(_rows([I] * 3, 400 * I, 4))
    want = duc_ref.definition_f64(h, y, incs, I, 999)
    assert np.abs(Q.definition_f64(h, list(y), incs, [I] * 3, 999) - want).max() <= 1e-12 * np.abs(want).max()
    got = Q.overlap_save_f64(h, list(y), incs, [I] * 3, 999)
    assert np.abs(got - want[:got.size]).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("Is,L,F", [([3, 5], 23, F_BIG), ([1], 7, 0), ([4, 8, 1], 64, F_TOP), ([2, 3], 1, 5),
                                    ([8, 10, 40], 255, 999)])
def test_adjoint_of_fcfb(Is, L, F):
    """<v, fcfb(x)> = <fcsb'(v), x> with fcsb' = (I_k = D_k, reversed taps, first_sample F - (L - 1), v followed by
    zero frames covering L - 1 positions) and x-hat read from position L - 1 on"""
    rng = np.random.default_rng(len(Is) + L)
    C_ = len(Is)
    incs = _incs(C_, L)
    h = rng.standard_normal((C_, L))
    Il = Q.lcm_of(Is)
    n = 37 * Il
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    v = [rng.standard_normal(n // I) + 1j * rng.standard_normal(n // I) for I in Is]
    Z = -(-(L - 1) // Il) * Il
    xh = Q.definition_f64(h[:, ::-1], [np.concatenate([vk, np.zeros(Z // I)]) for vk, I in zip(v, Is)], incs, Is,
                          (F - (L - 1)) % TWO64)
    y = fcfb_ref.definition_f64(h, x, incs, Is, F)
    lhs = sum(np.sum(np.conj(vk) * yk) for vk, yk in zip(v, y))
    rhs = np.sum(np.conj(xh[L - 1:L - 1 + n]) * x)
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs)


def round_trip_input(n, F, nus, bw, seed=10):
    """band-limited components (|f| < bw), component k mixed up to nus[k] by the exact NCO at absolute index F + n"""
    incs = [R.phase_increment_exact(nu, 1.0) for nu in nus]
    x = np.zeros(n, np.complex128)
    for k, inc in enumerate(incs):
        x += duc_ref.band_limited(n, bw, seed + k) * duc_ref.rot_up(R.phases(F, np.arange(n), inc))
    return x, incs


ROUND_TRIP = dict(Ds=[8, 8, 40], L=2561, nus=(-0.3, 0.05, 0.27), bw=0.004)


def test_round_trip_at_mixed_rates_reconstructs_the_input_f64():
    """fcfb(h_k, D_k) -> fcsb(f_k = D_k h_k, I_k = D_k, first_sample F - d): x[n - d], d = L - 1, with the drain of zero
    frames covering N positions"""
    Ds, L = ROUND_TRIP["Ds"], ROUND_TRIP["L"]
    h, f = Q.kaiser_pairs(Ds, L)
    n, F = 820 * 40, F_BIG
    x, incs = round_trip_input(n, F, ROUND_TRIP["nus"], ROUND_TRIP["bw"])
    y = fcfb_ref.definition_f64(h, x, incs, Ds, F)
    d = L - 1
    N, _ = Q.geometry(L, Ds)
    Il = Q.lcm_of(Ds)
    Z = -(-N // Il) * Il
    xr = Q.overlap_save_f64(f, [np.concatenate([yk, np.zeros(Z // D)]) for yk, D in zip(y, Ds)], incs, Ds,
                            (F - d) % TWO64)[:n]
    assert xr.size == n
    ref = x[2 * d:n - d]
    snr = 10 * np.log10(np.mean(np.abs(ref) ** 2) / np.mean(np.abs(xr[3 * d:] - ref) ** 2))
    print("f64 fcfb -> fcsb round trip: %.1f dB" % snr)
    assert snr >= ROUND_TRIP_SNR_DB, snr


def test_counts_and_drain_across_call_sequences():
    Is = [8, 10, 1, 40, 2]
    Il = Q.lcm_of(Is)
    N, P = Q.geometry(300, Is)
    for first in (0, 40 * 7 + 3, F_TOP):
        o0 = Q.off0(first, Is, P)
        rng = np.random.default_rng(first % 1000)
        total, got = 0, 0
        for step in list(rng.integers(0, 3 * P // Il, 40) * Il) + [Il] * 50 + [P, 0]:
            before = Q.counts(total, P, o0)
            total += int(step)
            got += Q.counts(total, P, o0) - before
        assert got == Q.counts(total, P, o0)
        assert total - P < got <= total
        # zero frames covering N positions (rounded up to Il) release every output of the stream
        assert Q.counts(total + -(-N // Il) * Il, P, o0) >= total


def _cfg(sdr, taps, n_taps, n_sets, inc, interp, C_):
    return sdr._ffi.FcsbConfig(taps.ctypes.data if taps is not None else None, n_taps, n_sets,
                               inc.ctypes.data if inc is not None else None,
                               interp.ctypes.data if interp is not None else None, C_, 0, 0, None)


def test_fcsb_argument_validation(sdr):
    L = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    inc = np.arange(4, dtype=np.uint64)
    interp = np.array([1, 2, 8, 10], np.uintp)
    zero = np.array([1, 0, 8, 10], np.uintp)
    many = np.zeros(257, np.uint64)
    many_i = np.ones(257, np.uintp)
    assert L.sdr_fcsb_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, inc, interp, 4),            # NULL taps
           _cfg(sdr, h, 64, 1, None, interp, 4),              # NULL increments
           _cfg(sdr, h, 64, 1, inc, None, 4),                 # NULL interpolations
           _cfg(sdr, h, 0, 1, inc, interp, 4),                # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, inc, interp, 4),    # L beyond 2^20
           _cfg(sdr, h, 64, 1, inc, interp, 0),               # C = 0
           _cfg(sdr, h, 64, 1, many, many_i, 257),            # beyond the channel limit
           _cfg(sdr, h, 64, 1, inc, zero, 4),                 # I_k = 0
           _cfg(sdr, h, 64, 2, inc, interp, 4),               # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 0, inc, interp, 4)]
    for cfg in bad:
        err.value = 0
        assert L.sdr_fcsb_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    nan = h.copy()
    nan[5] = np.inf
    err.value = 0
    assert L.sdr_fcsb_create(C.byref(_cfg(sdr, nan, 64, 1, inc, interp, 4)), C.byref(err)) is None
    assert err.value == 100
    huge = np.array([(1 << 22) + 1], np.uintp)                 # no N <= 2^22 fits
    err.value = 0
    assert L.sdr_fcsb_create(C.byref(_cfg(sdr, h, 64, 1, inc, huge, 1)), C.byref(err)) is None
    assert err.value == 101
    n = C.c_size_t(7)
    assert L.sdr_fcsb_process(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert L.sdr_fcsb_process_dev(None, None, 0, 0, None, 0, C.byref(n)) == 103
    assert L.sdr_fcsb_output_count(None, 100) == 0
    assert L.sdr_fcsb_reset(None) == 103
    assert L.sdr_fcsb_clone(None, C.byref(err)) is None and err.value == 103
    L.sdr_fcsb_destroy(None)


def test_fcsb_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Fcsb(gen.lowpass_taps(64, 0.05, 1.0), [100e3, -200e3], 2.4e6, [8, 10])
    assert e.value.code == 102

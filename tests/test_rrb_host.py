"""CPU: the rational resampler bank's computed form equals its definition (zero-stuff, np.convolve, keep (r+1) D - 1);
the reduction identity; cumulative counts; the zero-order-hold known answer; the oracle composition; argument
validation of sdr_rrb_create and the loud failure without a device."""
import ctypes as C
import math

import numpy as np
import pytest

import gen
import rrb_ref as R

# (I, D, L): I > L, D > L, I = D, gcd > 1, 1/1, I = 1, D = 1, 147/8000 and the ratios the bank is built for
CASES = [(I, D, L) for I, D in [(4, 25), (147, 160), (75, 64), (2, 25), (1, 5), (3, 4), (1, 1), (5, 1), (1, 7),
                                 (7, 7), (6, 4), (12, 18), (147, 8000), (16, 3), (40, 3)]
         for L in (1, 3, 17, 64)]


def _rows(n, seed):
    return gen.complex_noise(n, seed).astype(np.complex128)


@pytest.mark.parametrize("I,D,L", CASES)
def test_computed_form_equals_definition(I, D, L):
    h = np.random.default_rng(I * 31 + D + L).standard_normal(L)
    y = _rows(300 + D // I, I + D + L)
    want = R.definition_f64(h, y, I, D)
    got = R.computed_f64(h, y, I, D)
    assert got.shape == want.shape == (R.released(y.size, I, D),)
    if want.size:
        assert np.abs(got - want).max() <= 1e-12 * max(np.abs(want).max(), 1e-300)
        pick = np.array([0, want.size // 2, want.size - 1])
        assert np.abs(R.computed_f64(h, y, I, D, outputs=pick) - want[pick]).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("I,D,g,L", [(2, 3, 4, 50), (147, 160, 3, 3529), (1, 5, 7, 255), (4, 1, 5, 9), (1, 1, 6, 13),
                                     (3, 4, 2, 1)])
def test_reduction_has_the_same_chain(I, D, g, L):
    """(g I, g D, h) and (I, D, h[::g]): the same terms in the same order, hence the same f64 sums bit for bit"""
    h = np.random.default_rng(L).standard_normal(L)
    y = _rows(2000, g)
    r = np.arange(R.released(y.size, I, D))
    t1 = (r + 1) * D
    for (Ii, Di, hh) in ((g * I, g * D, h), (I, D, h[::g])):
        c, q = ((r + 1) * Di) % Ii, ((r + 1) * Di) // Ii
        assert np.array_equal(q, t1 // I)
        terms = [(hh[ci::Ii], q_) for ci, q_ in zip(c[:50], q[:50])]
        if Ii == g * I:
            full = terms
        else:
            for (a, qa), (b, qb) in zip(full, terms):
                assert qa == qb and np.array_equal(a, b)
    assert np.array_equal(R.computed_f64(h, y, g * I, g * D), R.computed_f64(h[::g], y, I, D))


@pytest.mark.parametrize("I,D", [(4, 25), (147, 160), (75, 64), (1, 1), (1, 5), (147, 8000), (6, 4)])
def test_counts_are_cumulative_floors(I, D):
    rng = np.random.default_rng(I + D)
    total, made = 0, 0
    for _ in range(200):
        n = int(rng.integers(0, 50))
        made += R.released(total + n, I, D) - R.released(total, I, D)
        total += n
        assert made == total * I // D
    # beyond 2^64 the exact count still holds
    big = (1 << 62) - 1
    assert R.released(big, 1 << 16, 3) == (big << 16) // 3 > (1 << 64)


@pytest.mark.parametrize("I,D", [(4, 25), (3, 4), (75, 64), (7, 2), (1, 3), (5, 1)])
def test_zero_order_hold_known_answer(I, D):
    """h = ones(I): z[r] = y[((r+1) D div I) - 1] exactly (y[-1] = 0 lies before the stream)"""
    y = _rows(500, I * D)
    z = R.computed_f64(np.ones(I), y, I, D)
    r = np.arange(z.size)
    assert np.array_equal(z, np.concatenate([[0], y])[((r + 1) * D) // I])


@pytest.mark.parametrize("I,D,L", [(4, 25, 101), (147, 160, 295), (3, 4, 17), (1, 5, 33), (5, 1, 10)])
def test_oracle_composition_matches_f64(I, D, L):
    h = gen.lowpass_taps(L, 0.4 / max(I, D), 1.0) * I
    y = _rows(400, L)
    z64 = R.computed_f64(h.astype(np.float32).astype(np.float64), y.astype(np.complex64), I, D)
    zo = R.oracle_f32(h, y, I, D)
    assert zo.shape == z64.shape
    assert np.abs(zo - z64).max() <= 1e-5 * np.abs(z64).max()


def test_shard_rule_prime_length():
    """H = a multiple of lcm(D_k / gcd) >= max ceil(L / I_k): the shard's first H I_k / D_k outputs cover its halo"""
    I, D, L = [4, 147, 75], [25, 160, 64], 1023
    step = math.lcm(*[d // math.gcd(i, d) for i, d in zip(I, D)])
    need = max(-(-L // i) for i in I)
    H = -(-need // step) * step
    for i, d in zip(I, D):
        assert (H * i) % d == 0


def _cfg(sdr, taps, L, sets, interp, decim, C_):
    return sdr._ffi.RrbConfig(None if taps is None else taps.ctypes.data, L, sets,
                              None if interp is None else interp.ctypes.data,
                              None if decim is None else decim.ctypes.data, C_, 0, None)


def test_rrb_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    one = np.ones(70000, np.uintp)
    bad_i = one.copy(); bad_i[2] = 0
    big_i = one.copy(); big_i[1] = (1 << 16) + 1
    bad_d = one.copy(); bad_d[3] = 0
    big_d = one.copy(); big_d[0] = (1 << 24) + 1
    assert lib.sdr_rrb_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, one, one, 4),             # NULL taps
           _cfg(sdr, h, 64, 1, None, one, 4),               # NULL interpolation
           _cfg(sdr, h, 64, 1, one, None, 4),               # NULL decimation
           _cfg(sdr, h, 0, 1, one, one, 4),                 # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, one, one, 4),     # L > 2^20
           _cfg(sdr, h, 64, 1, one, one, 0),                # C = 0
           _cfg(sdr, h, 64, 1, one, one, 65537),            # C > 65536
           _cfg(sdr, h, 64, 2, one, one, 4),                # n_tap_sets not in {1, C}
           _cfg(sdr, h, 1 << 20, 65536, one, one, 65536),   # n_tap_sets * n_taps > 2^26
           _cfg(sdr, h, 64, 1, bad_i, one, 4),              # I = 0
           _cfg(sdr, h, 64, 1, big_i, one, 4),              # I > 2^16
           _cfg(sdr, h, 64, 1, one, bad_d, 4),              # D = 0
           _cfg(sdr, h, 64, 1, one, big_d, 4)]              # D > 2^24
    for cfg in bad:
        err.value = 0
        assert lib.sdr_rrb_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    n = np.zeros(4, np.uintp)
    assert lib.sdr_rrb_process(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_rrb_process_dev(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_rrb_output_count(None, n.ctypes.data, n.ctypes.data) == 103
    assert lib.sdr_rrb_reset(None) == 103
    assert lib.sdr_rrb_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_rrb_destroy(None)


def test_rrb_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Rrb(gen.lowpass_taps(64, 1.0 / 25, 4.0), 4, 25, n_channels=3)
    assert e.value.code == 102

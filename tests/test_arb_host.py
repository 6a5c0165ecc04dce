"""CPU: the arbitrary-ratio resampler bank's computed form equals its literal definition (exact weights) and stays
within the truncation bound (the kernel's 2^-24 weights); the exact relation to sdr_rrb's definition; exact counts over
blockings and across set_steps; sdr_arb_step's rounding; argument validation and the handle lifecycle without a device."""
import ctypes as C
import itertools
from fractions import Fraction

import numpy as np
import pytest

import arb_ref as A
import gen
import rrb_ref

ONE = A.ONE

# steps in units of 2^-64: ppm offsets, 48000/44100 and its inverse, 6.25 (1 + 37e-6), 1/4.41, the range ends, 1
STEPS = [ONE + ONE * 37 // 1000000, ONE - ONE * 37 // 1000000, A.step_of(48000.0, 44100.0), A.step_of(44100.0, 48000.0),
         A.step_of(6.25 * (1 + 37e-6), 1.0), A.step_of(1.0, 4.41), 1 << 48, 3 * ONE + 12345, ONE]
FIRSTS = [0, (17 << 64) | 0x9E3779B97F4A7C15, 0x00000000FFFFFFFF, (1 << 40 << 64) + (5 << 60)]
CASES = [(P, L, s, f) for (P, L), s, f in zip(itertools.cycle([(1, 1), (1, 7), (2, 7), (8, 33), (32, 255), (256, 255),
                                                                (4, 1), (256, 4096), (16, 100), (64, 65)]),
                                              STEPS * 7, itertools.cycle(FIRSTS))]


def _window(first, step, L, P, n_out):
    """exact positions of n_out outputs and a row that covers their windows, starting at absolute frame `at`"""
    taus = [first + r * step for r in range(n_out)]
    at = max(0, (taus[0] >> 64) - L // P - 4)
    n = (taus[-1] >> 64) - at + 1
    return taus, at, n


@pytest.mark.parametrize("P,L,step,first", CASES)
def test_computed_form_equals_definition(P, L, step, first):
    assert len(CASES) >= 60
    rng = np.random.default_rng(P * 7 + L + (step & 0xFFFF))
    h = rng.standard_normal(L)
    taus, at, n = _window(first, step, L, P, 24)
    y = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    want = A.definition_f64(h, P, y, taus, at=at)
    got = A.computed_f64(h, P, y, taus, at=at)
    scale = max(np.abs(want).max(), 1e-300)
    assert np.abs(got - want).max() <= 1e-12 * scale
    trunc, sad = A.computed_f64(h, P, y, taus, at=at, truncated=True, bound=True)
    assert (np.abs(trunc - got) <= 2.0 ** -24 * sad + 1e-12 * scale).all()


@pytest.mark.parametrize("I,D,L", [(2, 3, 9), (8, 5, 33), (32, 147, 255), (8, 1, 17), (2, 25, 64), (32, 31, 100)])
def test_rrb_relation(I, D, L):
    """P = I, sigma = D / I, tau(0) = ((r0+1) D - I) / I: sdr_rrb's outputs r >= r0 (the first r0 are 0), and the
    count differs by the outputs whose tau lies in (n-1, n)"""
    rng = np.random.default_rng(I + D + L)
    h = rng.standard_normal(L)
    n = 200 + 3 * L
    y = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    r0, first = A.rrb_first(I, D)
    step = D * ONE // I
    assert step * I == D * ONE and first * I == ((r0 + 1) * D - I) * ONE
    zr = rrb_ref.definition_f64(h, y, I, D)
    assert (zr[:r0] == 0).all()
    cnt = A.released(n, first, step)
    taus = [first + r * step for r in range(cnt)]
    za = A.definition_f64(h, I, y, taus)
    common = min(za.size, zr.size - r0)
    assert common > 0
    assert np.abs(za[:common] - zr[r0:r0 + common]).max() <= 1e-12 * np.abs(zr).max()
    # the weights are 0 on this grid, so the computed form holds the same terms as sdr_rrb's chain
    assert all(x == 0 for x in A._split(taus, I)[2])
    for m in range(0, n, 7):
        arb_n, rrb_n = A.released(m, first, step), max(0, rrb_ref.released(m, I, D) - r0)
        early = sum(1 for r in range(rrb_n, arb_n + 2) if (m - 1) * ONE < first + r * step < m * ONE)
        assert arb_n - rrb_n == early, m


@pytest.mark.parametrize("step,first", [(s, f) for s in STEPS[:7] for f in FIRSTS[:3]])
def test_counts_brute_force_and_blockings(step, first):
    taus = [first + r * step for r in range(4000)]
    for n in list(range(0, 40)) + [int(x) for x in np.random.default_rng(step & 0xFFFF).integers(0, 300, 30)]:
        if n * ONE > taus[-1]:
            continue
        assert A.released(n, first, step) == sum(1 for t in taus if t < n * ONE)
    rng = np.random.default_rng(first & 0xFFFF)
    total, made = 0, 0
    for _ in range(300):
        k = int(rng.integers(0, 20))
        made += A.released(total + k, first, step) - A.released(total, first, step)
        total += k
        assert made == A.released(total, first, step)


def test_counts_across_set_steps():
    """per-call counts over random blockings with steps changed between calls add up to #{r : tau(r) < n}"""
    rng = np.random.default_rng(3)
    steps = [s for s in STEPS if s >= ONE // 8]  # the brute force walks every output
    for trial in range(20):
        tb = A.Timebase(int(rng.integers(0, 1 << 62)) * 20, steps[trial % len(steps)])
        total, made = 0, 0
        for call in range(60):
            if call % 7 == 3:
                tb.set_step(total, steps[int(rng.integers(0, len(steps)))])
            k = int(rng.integers(0, 50))
            made += tb.released(total + k) - tb.released(total)
            total += k
            # brute force over the piecewise positions
            r = 0
            while tb.tau(r) < total * ONE:
                r += 1
            assert made == r
        # the positions before a change are the old ones; after it they advance by the new step
        for (rb, base, st), (rb2, base2, _) in zip(tb.segs, tb.segs[1:]):
            assert base2 == base + (rb2 - rb) * st


def test_arb_step_rounding(sdr):
    lib = sdr.lib()
    t = sdr._ffi.ArbTime()
    pairs = [(48000.0, 44100.0), (44100.0, 48000.0), (1.000037, 1.0), (6.25 * (1 + 37e-6), 1.0), (1.0, 4.41),
             (2.048e6, 48000.0), (1.0, 65536.0), (16777216.0, 1.0), (3.0, 7.0), (1.0, 3.0), (0.1, 0.3), (1e300, 1e299),
             (5e-324, 5e-324), (np.nextafter(1.0, 2.0), 1.0)]
    rng = np.random.default_rng(4)
    pairs += [(float(a), float(b)) for a, b in zip(np.exp(rng.uniform(-5, 5, 40)), np.exp(rng.uniform(-5, 5, 40)))]
    # ties: quotients with exactly one bit below 2^-64 (only possible for sigma < 2^-12: a double has 53 bits)
    ties = [(((1 << 50) + 1) * 2.0 ** -65, 1.0), (((1 << 50) + 3) * 2.0 ** -65, 1.0),
            (3.0 * ((1 << 49) + 1) * 2.0 ** -65, 3.0)]
    pairs += ties
    for a, b in pairs:
        want = A.step_of(float(a), float(b))
        rc = lib.sdr_arb_step(float(a), float(b), C.byref(t))
        if want is None:
            assert rc == 100, (a, b)
        else:
            assert rc == 0 and (t.whole << 64 | t.frac) == want, (a, b)
            assert sdr.arb_step(a, b) == want
    for a, b in ties:
        q = Fraction(a) / Fraction(b) * ONE
        assert q.denominator == 2 and A.step_of(a, b) % 2 == 0
    for a, b in [(0.0, 1.0), (-1.0, 1.0), (1.0, 0.0), (float("nan"), 1.0), (float("inf"), 1.0), (1.0, float("inf")),
                 (1.0, 65537.0), (2.0 ** 24 + 1, 1.0), (1.0, 1e30)]:
        assert lib.sdr_arb_step(a, b, C.byref(t)) == 100, (a, b)
    assert lib.sdr_arb_step(1.0, 1.0, None) == 4


def _cfg(sdr, taps, L, sets, P, steps, first, C_):
    return sdr._ffi.ArbConfig(None if taps is None else taps.ctypes.data, L, sets, P,
                              None if steps is None else C.addressof(steps),
                              None if first is None else C.addressof(first), C_, 0, None)


def _times(sdr, vals):
    return (sdr._ffi.ArbTime * len(vals))(*[sdr._ffi.ArbTime(v >> 64, v & (ONE - 1)) for v in vals])


def test_arb_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    st = _times(sdr, [ONE] * 4)
    lo = _times(sdr, [ONE] * 3 + [(1 << 48) - 1])
    hi = _times(sdr, [(1 << 88) + 1] + [ONE] * 3)
    fz = _times(sdr, [0] * 4)
    far = _times(sdr, [0, 0, 1 << 62 << 64, 0])
    assert lib.sdr_arb_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, 8, st, None, 4),            # NULL taps
           _cfg(sdr, h, 64, 1, 8, None, None, 4),             # NULL steps
           _cfg(sdr, h, 64, 1, 0, st, None, 4),               # P = 0
           _cfg(sdr, h, 64, 1, 12, st, None, 4),              # P not a power of two
           _cfg(sdr, h, 64, 1, 1 << 17, st, None, 4),         # P > 2^16
           _cfg(sdr, h, 0, 1, 8, st, None, 4),                # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, 8, st, None, 4),    # L > 2^20
           _cfg(sdr, h, 64, 1, 8, st, None, 0),               # C = 0
           _cfg(sdr, h, 64, 2, 8, st, None, 4),               # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 1, 8, lo, None, 4),               # sigma < 2^-16
           _cfg(sdr, h, 64, 1, 8, hi, None, 4),               # sigma > 2^24
           _cfg(sdr, h, 64, 1, 8, st, far, 4)]                # first whole part >= 2^62
    for cfg in bad:
        err.value = 0
        assert lib.sdr_arb_create(C.byref(cfg), C.byref(err)) is None and err.value == 100
    many = _times(sdr, [ONE] * 65537)
    err.value = 0
    assert lib.sdr_arb_create(C.byref(_cfg(sdr, h, 64, 1, 8, many, None, 65537)), C.byref(err)) is None
    assert err.value == 100                                    # C > 65536
    n = np.zeros(4, np.uintp)
    assert lib.sdr_arb_process(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_arb_process_dev(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_arb_output_count(None, n.ctypes.data, n.ctypes.data) == 103
    assert lib.sdr_arb_reset(None) == 103
    assert lib.sdr_arb_set_steps(None, C.addressof(st)) == 103
    assert lib.sdr_arb_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_arb_destroy(None)
    if sdr.device_count() == 0:
        err.value = 0
        assert lib.sdr_arb_create(C.byref(_cfg(sdr, h, 64, 1, 8, st, fz, 4)), C.byref(err)) is None
        assert err.value == 102


def test_arb_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Arb(gen.lowpass_taps(256, 0.4, 32.0) * 32, 32, sdr.arb_step(48000, 44100), n_channels=3)
    assert e.value.code == 102

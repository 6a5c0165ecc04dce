"""CPU: the symbol timing recovery bank's reference model (tsync_ref) and ABI without a device.  The loop-design helper
equals its closed form; create rejects every invalid parameter and fails with NO_DEVICE for a valid one; NULL handles
give NULL_HANDLE.  The model with kp = ki = 0 is sdr_arb's (positions, counts and interpolant); its count bound holds
over random trajectories and blockings; with gains from the loop design it acquires and tracks RRC-shaped QPSK at the
bars the GPU tests use (the sign of the corrections is checked here)."""
import ctypes as C

import numpy as np
import pytest

import arb_ref as A
import tsync_ref as R

ONE = A.ONE
F32 = np.float32

# the tracking bars of test_gpu_tsync.py, after ACQ symbols: set from this model's runs (worst over 64 channels:
# 0.030 T, EVM 0.036, 4.9 ppm) with margin
ACQ = 1000
BAR_TIMING, BAR_EVM, BAR_PPM = 0.06, 0.06, 20e-6


def test_loop_design_closed_form(sdr):
    for bn, z, k, t in [(0.01, 0.707, 1.078, 4.0), (0.005, 1.0, 2.0, 2.000074), (0.05, 0.5, 0.3, 8.25),
                        (1e-4, 0.707, 1.0, 1.0), (0.2, 2.0, 5.0, 1 << 20)]:
        kp, ki = sdr.tsync_loop_design(bn, z, k, t)
        th = bn / (z + 1 / (4 * z))
        d = 1 + 2 * z * th + th * th
        assert kp == F32(4 * z * th / (d * k) * t) and ki == F32(4 * th * th / (d * k) * t)
        assert (kp, ki) == tuple(F32(x) for x in R.loop_design(bn, z, k, t))
    lib = sdr.lib()
    a, b = C.c_float(), C.c_float()
    for bad in [(0.0, 0.7, 1.0, 4.0), (0.01, -1.0, 1.0, 4.0), (0.01, 0.7, 0.0, 4.0), (0.01, 0.7, 1.0, float("inf")),
                (float("nan"), 0.7, 1.0, 4.0)]:
        assert lib.sdr_tsync_loop_design(*bad, C.byref(a), C.byref(b)) == 100, bad
    assert lib.sdr_tsync_loop_design(0.01, 0.7, 1.0, 4.0, None, C.byref(b)) == 4


def _times(sdr, vals):
    return (sdr._ffi.ArbTime * len(vals))(*[sdr._ffi.ArbTime(v >> 64, v & (ONE - 1)) for v in vals])


def _loops(sdr, loops):
    return (sdr._ffi.TsyncLoop * len(loops))(*[sdr._ffi.TsyncLoop(*x) for x in loops])


def _cfg(sdr, taps, L, sets, P, periods, first, loops, n_loops, C_):
    """the config keeps its arrays alive"""
    cfg = sdr._ffi.TsyncConfig(None if taps is None else taps.ctypes.data, L, sets, P,
                                None if periods is None else C.addressof(periods),
                                None if first is None else C.addressof(first),
                                None if loops is None else C.addressof(loops), n_loops, C_, 0, None)
    cfg.keep = (taps, periods, first, loops)
    return cfg


def test_tsync_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    h = np.ones(4 * 64, np.float32)
    T4 = 4 * ONE
    per = _times(sdr, [T4] * 4)
    ok = _loops(sdr, [(0.05, 0.001, 1.0, 0.01)])
    bad_periods = [[T4] * 3 + [ONE - 1], [T4] * 3 + [(1 << 84) + 1]]
    bad_loops = [(0.05, 0.001, 1.0, 0.26), (0.05, 0.001, 1.0, -1e-9), (0.05, 0.001, 1.0, float("nan")),
                 (-0.05, 0.001, 1.0, 0.01), (0.05, -0.001, 1.0, 0.01), (float("inf"), 0.0, 1.0, 0.01),
                 (0.05, float("nan"), 1.0, 0.01), (0.05, 0.001, 0.0, 0.01), (0.05, 0.001, -1.0, 0.01),
                 (0.05, 0.001, float("inf"), 0.01),
                 (0.0, 2.0 ** 22, 1.0, 0.01),     # fl(ki err_max) >= 2^22 frames
                 (1.0, 0.0, 1.0, 0.0),            # at T = 2 frames: 2 D = 2 frames = T - V
                 (0.99, 0.0, 2.0, 0.01)]          # at T = 4 frames: 2 D = 2 fl(0.99 * 2) > T - V = 3.96
    assert lib.sdr_tsync_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, None, 64, 1, 8, per, None, ok, 1, 4),             # NULL taps
           _cfg(sdr, h, 64, 1, 8, None, None, ok, 1, 4),               # NULL periods
           _cfg(sdr, h, 64, 1, 8, per, None, None, 1, 4),              # NULL loops
           _cfg(sdr, h, 64, 1, 8, per, None, ok, 2, 4),                # n_loops not in {1, C}
           _cfg(sdr, h, 64, 1, 0, per, None, ok, 1, 4),                # P = 0
           _cfg(sdr, h, 64, 1, 12, per, None, ok, 1, 4),               # P not a power of two
           _cfg(sdr, h, 64, 1, 1 << 17, per, None, ok, 1, 4),          # P > 2^16
           _cfg(sdr, h, 0, 1, 8, per, None, ok, 1, 4),                 # L = 0
           _cfg(sdr, h, (1 << 20) + 1, 1, 8, per, None, ok, 1, 4),     # L > 2^20
           _cfg(sdr, h, 64, 1, 8, per, None, ok, 1, 0),                # C = 0
           _cfg(sdr, h, 64, 2, 8, per, None, ok, 1, 4),                # n_tap_sets not in {1, C}
           _cfg(sdr, h, 64, 1, 8, per, _times(sdr, [0, 0, 1 << 62 << 64, 0]), ok, 1, 4)]  # first whole >= 2^62
    bad += [_cfg(sdr, h, 64, 1, 8, _times(sdr, p), None, ok, 1, 4) for p in bad_periods]
    loops_t = [None] * len(bad_loops)
    for i, lp in enumerate(bad_loops):
        T = 2 * ONE if i == len(bad_loops) - 2 else T4
        loops_t[i] = _loops(sdr, [(0.05, 0.001, 1.0, 0.01)] * 3 + [lp])
        bad.append(_cfg(sdr, h, 64, 1, 8, _times(sdr, [T] * 4), None, loops_t[i], 4, 4))
    assert not R.valid(2 * ONE, bad_loops[-2]) and not R.valid(T4, bad_loops[-1])
    assert R.valid(2 * ONE, (0.999, 0.0, 1.0, 0.0)) and R.valid(T4, (0.98, 0.0, 2.0, 0.01))
    for i, cfg in enumerate(bad):
        err.value = 0
        assert lib.sdr_tsync_create(C.byref(cfg), C.byref(err)) is None and err.value == 100, i
    many = _times(sdr, [T4] * 65537)
    err.value = 0
    assert lib.sdr_tsync_create(C.byref(_cfg(sdr, h, 64, 1, 8, many, None, ok, 1, 65537)), C.byref(err)) is None
    assert err.value == 100                                              # C > 65536
    n = np.zeros(4, np.uintp)
    t, v = sdr._ffi.ArbTime(), C.c_int64()
    assert lib.sdr_tsync_process(None, None, n.ctypes.data, 0, None, None, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_tsync_process_dev(None, None, n.ctypes.data, 0, None, None, None, 0, 0, n.ctypes.data) == 103
    assert lib.sdr_tsync_max_output(None, n.ctypes.data, n.ctypes.data) == 103
    assert lib.sdr_tsync_get_state(None, 0, C.byref(t), C.byref(v)) == 103
    assert lib.sdr_tsync_reset(None) == 103
    assert lib.sdr_tsync_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_tsync_destroy(None)
    if sdr.device_count() == 0:
        # valid, at the edges: T = 1 and 2^20 frames, max_dev = 0.25, per-channel loops
        edge = _loops(sdr, [(0.05, 0.001, 1.0, 0.25), (0.0, 0.0, 1.0, 0.0), (0.1, 0.0, 1.0, 0.01),
                            (0.05, 0.001, 1.0, 0.01)])
        err.value = 0
        cfg = _cfg(sdr, h, 64, 1, 8, _times(sdr, [ONE, 1 << 84, T4, T4]), _times(sdr, [0, 5, ONE // 3, 7 << 64]),
                   edge, 4, 4)
        assert lib.sdr_tsync_create(C.byref(cfg), C.byref(err)) is None and err.value == 102


def test_tsync_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Tsync(np.ones(33, np.float32), 8, 4 * ONE, (0.05, 0.001, 1.0, 0.01), n_channels=3)
    assert e.value.code == 102


def test_dev_bound_is_exact():
    for md in (0.0, 0.25, 0.01, 100e-6, 5e-324, 0.1, 1e-300):
        for T in (ONE, 1 << 84, A.step_of(4.41, 1.0), A.step_of(2 * (1 + 37e-6), 1.0)):
            V = R.dev_bound(md, T)
            from fractions import Fraction
            exact = Fraction(md) * T / (1 << 24)
            assert V <= exact < V + 1


@pytest.mark.parametrize("P,L,T,first", [(1, 1, 2 * ONE, 0), (32, 255, A.step_of(4.41, 1.0), (3 << 64) + 12345),
                                         (8, 65, A.step_of(2 * (1 + 37e-6), 1.0), ONE // 3),
                                         (256, 2049, A.step_of(10.3, 1.0), 0)])
def test_model_open_loop_is_arb(P, L, T, first):
    """kp = ki = 0: positions first + r T, sdr_arb's counts, and y = sdr_arb's computed form (truncated weights)"""
    rng = np.random.default_rng(L)
    h = rng.standard_normal(L)
    n = 700
    y = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    ys, pos, es, vs = R.model(h, P, y, T, (0.0, 0.0, 1.0, 0.01), first=first)
    assert len(ys) == A.released(n, first, T)
    assert pos == [first + r * T for r in range(len(ys))]
    assert set(vs) == {0} and es[0] == 0
    z = A.computed_f64(h, P, y, pos, truncated=True)
    assert np.array_equal(ys, z.astype(np.complex64))
    # and the replay of the model's own errors gives its positions
    vs2, _ = R.replay(pos, es, T, (0.0, 0.0, 1.0, 0.01), first=first)
    assert vs2 == vs


@pytest.mark.parametrize("seed", range(6))
def test_model_bound_never_exceeded(seed):
    """aggressive loops (corrections up to the validity limit) on noise: for random blockings, the symbols a call
    releases never exceed max_output, and replay reproduces the model's positions"""
    rng = np.random.default_rng(seed)
    period = [2.0, 2 * (1 + 37e-6), 4.41, 8.0, 10.3, 1.0][seed]
    T = A.step_of(period, 1.0)
    md = [0.25, 0.01, 0.1, 0.0, 0.2, 0.05][seed]
    emax = 1.5
    kp = F32(0.49 * (1 - md) * period / emax)  # 2 D just below T - V
    loop = (kp, F32(0.02 * period), F32(emax), md)
    assert R.valid(T, loop)
    n = 3000
    y = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64) * 2
    h = rng.standard_normal(17)
    ys, pos, es, vs = R.model(h, 4, y, T, loop, first=int(rng.integers(0, 1 << 62)) * 12)
    steps = np.diff(np.array(pos, dtype=object))
    assert min(steps) >= R.t_min(T, loop) > 0
    assert (np.abs(es) > 0).mean() > 0.9
    vs2, _ = R.replay(pos, es, T, loop)
    assert vs2 == vs
    total = 0
    while total < n:
        k = int(rng.integers(0, 60))
        got = sum(1 for t in pos if total <= (t >> 64) < total + k)
        assert got <= R.max_output(k, T, loop), (total, k)
        total += k


def test_model_acquires_and_tracks_qpsk():
    """RRC QPSK (beta = 0.35, span 8) at 2-8 frames per symbol, clock offsets 0, +-50, +-500 ppm, random delays,
    Es/N0 = 30 dB; gains from the loop design (B_n T = 0.01, zeta = 0.707) and the Gardner slope of the RC pulse"""
    beta, span, P = 0.35, 8, 32
    K = R.gardner_slope(beta)
    rng = np.random.default_rng(2)
    for i, (period, ppm) in enumerate([(2, 0), (2.5, 50e-6), (3, -50e-6), (4, 500e-6), (8, -500e-6), (6, 0),
                                       (5, 500e-6), (2, -500e-6)]):
        true = period * (1 + ppm)
        T = A.step_of(period, 1.0)
        kp, ki = R.loop_design(0.01, 0.707, K, period)
        loop = (F32(kp), F32(ki), 2.0, 0.01)
        d = rng.uniform(0, true)
        y, _ = R.qpsk_channel(int(3000 * true), true, d, beta, span, 30.0, rng)
        h, c = R.rrc_taps(period, P, beta, span)
        ys, pos, es, vs = R.model(h, P, y, T, loop)
        timing, evm, dppm = R.tracking(pos, ys, vs, T, true, d, c, ACQ)
        assert timing < BAR_TIMING and evm < BAR_EVM and abs(dppm) < BAR_PPM, (period, ppm, timing, evm, dppm)

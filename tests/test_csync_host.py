"""CPU: the carrier recovery bank's reference model (csync_ref) and ABI without a device.  create rejects every invalid
parameter and fails with NO_DEVICE for a valid one; NULL handles give NULL_HANDLE.  sdr_tsync_loop_design with a period
of 1 / (2 pi) is the type-2 loop in turns; the detector slopes K_d of the header's table hold numerically; the open loop
advances the phase by exactly 2^24 nu_0 per symbol; replay reproduces the model's phases; with gains from the loop
design the model acquires and tracks BPSK, QPSK and 8PSK at known offsets and phases at the bars the GPU tests use (the
sign of the corrections is checked here)."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

import csync_ref as R

F32 = np.float32

# the tracking workload and bars of test_gpu_csync.py: Es/N0 = 30 dB, B_n T = 0.01, zeta = 0.707, offsets in turns per
# symbol, ACQ of N symbols skipped.  Set from this model's runs (worst over 64 channels per order: RMS phase error
# 0.0042 rad, EVM 0.0326, |nu - f| 2.7e-5 turn per symbol) with margin.
OFFSETS = [0.0, 1e-4, -1e-4, 2e-3, -2e-3]
N, ACQ = 4000, 1000
ESN0, BN_T, ZETA, ERR_MAX, MAX_FREQ = 30.0, 0.01, 0.707, 2.0, 0.01
BAR_PHASE, BAR_EVM, BAR_FREQ = 0.01, 0.05, 1e-4
KD = {2: 1.0, 4: np.sqrt(2.0), 8: 1.0 / np.cos(np.pi / 8)}


def design(sdr, M, A=1.0):
    """the loop of the tracking workload for order M at amplitude A, gains from sdr_tsync_loop_design"""
    kp, ki = sdr.tsync_loop_design(BN_T, ZETA, KD[M] * A, 1 / (2 * np.pi))
    return (M, kp, ki, ERR_MAX, MAX_FREQ)


def test_loop_design_in_turns(sdr):
    for bn, z, M in [(0.01, 0.707, 2), (0.005, 1.0, 4), (0.05, 0.5, 8), (1e-4, 0.707, 4)]:
        kp, ki = sdr.tsync_loop_design(bn, z, KD[M], 1 / (2 * np.pi))
        th = bn / (z + 1 / (4 * z))
        d = 1 + 2 * z * th + th * th
        assert kp == F32(4 * z * th / (d * KD[M]) / (2 * np.pi)) and ki == F32(4 * th * th / (d * KD[M]) / (2 * np.pi))
        assert (kp, ki) == tuple(F32(x) for x in R.loop_design(bn, z, KD[M]))


@pytest.mark.parametrize("M", [2, 4, 8])
def test_detector_slope(M):
    """K_d = A, sqrt(2) A, A / cos(pi / 8): the mean detector output per radian at zero phase error"""
    for A in (0.25, 1.0, 3.0):
        assert abs(R.slope(M, A) - KD[M] * A) < 1e-6 * KD[M] * A


def test_detector_float32_cases():
    """signs of zeros, the M = 8 branch boundary, and non-finite inputs"""
    zr = np.array([0.0, -0.0, 1.0, -1.0, 0.5, np.nan, np.inf, 2.0], F32)
    zi = np.array([-0.0, 0.0, 1.0, 1.0, -0.25, 1.0, 1.0, -2.0], F32)
    assert np.array_equal(R.detector(zr, zi, 2), np.array([-0.0, 0.0, 1, -1, -0.25, -1, 1, -2], F32))
    a = np.where(zr >= 0, zi, -zi)
    b = np.where(zi >= 0, zr, -zr)
    with np.errstate(invalid="ignore"):
        assert np.array_equal(R.detector(zr, zi, 4), a - b, equal_nan=True)
        g8 = R.detector(zr, zi, 8)
    assert g8[2] == F32(1) - R.K8 * F32(1) and g8[7] == F32(-2) - R.K8 * F32(-2)  # |re| = |im|: the first branch
    assert g8[4] == F32(-0.25) - R.K8 * F32(-0.5)
    e = R.clamp_err(np.array([np.nan, np.inf, -np.inf, 5.0, -5.0, 0.5], F32), 2.0)
    assert np.array_equal(e, np.array([0, 0, 0, 2, -2, 0.5], F32))


def test_dev_bound_is_exact():
    for f in (0.0, 0.25, 1 / 16, 0.01, 1e-3, 5e-324, 0.1, 1e-300):
        V = R.dev_bound(f)
        assert V <= Fraction(f) * 2 ** 40 < V + 1


def _cfg(sdr, loops, C_, phase=None, freq=None, n_loops=None):
    """the config keeps its arrays alive"""
    lp = (sdr._ffi.CsyncLoop * len(loops))(*[sdr._ffi.CsyncLoop(*x) for x in loops]) if loops is not None else None
    ph = None if phase is None else (C.c_uint64 * len(phase))(*phase)
    fr = None if freq is None else (C.c_int64 * len(freq))(*freq)
    cfg = sdr._ffi.CsyncConfig(None if lp is None else C.addressof(lp), len(loops) if n_loops is None else n_loops,
                               None if ph is None else C.addressof(ph), None if fr is None else C.addressof(fr), C_,
                               0, None)
    cfg.keep = (lp, ph, fr)
    return cfg


def test_csync_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    ok = (4, 0.004, 3e-5, 2.0, 0.01)
    bad_loops = [(3, 0.004, 3e-5, 2.0, 0.01), (0, 0.004, 3e-5, 2.0, 0.01), (16, 0.004, 3e-5, 2.0, 0.01),
                 (4, -0.004, 3e-5, 2.0, 0.01), (4, 0.004, -3e-5, 2.0, 0.01), (4, float("inf"), 0.0, 2.0, 0.01),
                 (4, float("nan"), 0.0, 2.0, 0.01), (4, 0.0, float("nan"), 2.0, 0.01),
                 (4, 0.004, 3e-5, 0.0, 0.01), (4, 0.004, 3e-5, -1.0, 0.01), (4, 0.004, 3e-5, float("inf"), 0.01),
                 (4, 0.004, 3e-5, float("nan"), 0.01),
                 (4, 0.0625, 0.0, 2.0, 0.01),     # fl(kp err_max) = 1/8 = 1/(2M)
                 (8, 0.0, 0.03125, 2.0, 0.01),    # fl(ki err_max) = 1/16 = 1/(2M)
                 (2, 0.125, 0.0, 2.0, 0.01),      # fl(kp err_max) = 1/4 = 1/(2M)
                 (4, 0.004, 3e-5, 2.0, -1e-9), (4, 0.004, 3e-5, 2.0, 0.125 + 1e-12),
                 (8, 0.004, 3e-5, 2.0, 1 / 16 + 1e-12), (4, 0.004, 3e-5, 2.0, float("nan"))]
    assert lib.sdr_csync_create(None, C.byref(err)) is None and err.value == 100
    V = R.dev_bound(0.01)
    bad = [_cfg(sdr, None, 4, n_loops=1),                              # NULL loops
           _cfg(sdr, [ok, ok], 4),                                     # n_loops not in {1, C}
           _cfg(sdr, [ok], 0),                                         # C = 0
           _cfg(sdr, [ok], 4, freq=[0, V + 1, 0, 0]),                  # nu_0 > V
           _cfg(sdr, [ok], 4, freq=[0, 0, 0, -V - 1]),                 # nu_0 < -V
           _cfg(sdr, [(4, 0.004, 3e-5, 2.0, 0.0)], 2, freq=[0, 1])]    # V = 0
    bad += [_cfg(sdr, [ok] * 3 + [lp], 4) for lp in bad_loops]
    for i, cfg in enumerate(bad):
        err.value = 0
        assert lib.sdr_csync_create(C.byref(cfg), C.byref(err)) is None and err.value == 100, i
    err.value = 0
    assert lib.sdr_csync_create(C.byref(_cfg(sdr, [ok], 65537)), C.byref(err)) is None and err.value == 100
    n = np.zeros(4, np.uintp)
    ph, fr = C.c_uint64(), C.c_int64()
    assert lib.sdr_csync_process(None, None, n.ctypes.data, 0, None, None, None, 0) == 103
    assert lib.sdr_csync_process_dev(None, None, n.ctypes.data, 0, None, None, None, 0) == 103
    assert lib.sdr_csync_get_state(None, 0, C.byref(ph), C.byref(fr)) == 103
    assert lib.sdr_csync_reset(None) == 103
    assert lib.sdr_csync_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_csync_destroy(None)
    if sdr.device_count() == 0:
        # valid, at the edges: every order, the largest corrections and frequency ranges, nu_0 = +-V, C = 65536
        edge = [(2, 0.12499, 0.0, 2.0, 0.25), (4, 0.0, 0.06249, 2.0, 0.125), (8, 0.0312, 0.0312, 2.0, 1 / 16),
                (4, 0.0, 0.0, 1e-30, 0.0)]
        for cfg in [_cfg(sdr, edge, 4, phase=[0, 1 << 63, (1 << 64) - 1, 5],
                         freq=[R.dev_bound(0.25), -R.dev_bound(0.125), R.dev_bound(1 / 16), 0]),
                    _cfg(sdr, [ok], 65536)]:
            err.value = 0
            assert lib.sdr_csync_create(C.byref(cfg), C.byref(err)) is None and err.value == 102


def test_csync_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Csync((4, 0.004, 3e-5, 2.0, 0.01), n_channels=3)
    assert e.value.code == 102


def test_model_open_loop_and_replay():
    """kp = ki = 0: phi_s = phi_0 + s 2^24 nu_0 (mod 2^64) exactly and z = x e^{-2 pi i phi_s / 2^64}; replay of the
    model's own errors gives its phases, with a closed loop and per-channel orders"""
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((3, 300)) + 1j * rng.standard_normal((3, 300))).astype(np.complex64)
    phi0 = [0, 1 << 63, int(rng.integers(0, 1 << 63)) * 2 + 1]
    nu0 = [0, R.dev_bound(0.01), -12345]
    z, ph, e, nu = R.model(x, (4, 0.0, 0.0, 2.0, 0.01), phi0, nu0)
    for k in range(3):
        assert [int(p) for p in ph[k]] == [(phi0[k] + s * (nu0[k] << 24)) % (1 << 64) for s in range(300)]
        assert (nu[k] == nu0[k]).all()
    assert np.abs(z - R.rotate(x, ph)).max() < 1e-6 * np.abs(x).max()
    loops = [(2, 0.01, 1e-4, 1.0, 0.05), (4, 0.02, 2e-3, 2.0, 0.01), (8, 0.03, 3e-4, 0.5, 1 / 16)]
    z, ph, e, nu = R.model(x * 3, loops, phi0, [0, 0, 5])
    assert (np.abs(e) > 0).mean() > 0.9
    nus, (phi_n, nu_n) = R.replay(ph, e, [300] * 3, loops, phi0, [0, 0, 5])
    assert np.array_equal(nus, nu)
    want = R.Loops(loops, 3).step(ph[:, -1], nu[:, -1], e[:, -1])
    assert np.array_equal(phi_n, want[0]) and np.array_equal(nu_n, want[1])
    # the frequency never leaves [-V, V]
    assert all(np.abs(nu[k]).max() <= R.dev_bound(loops[k][4]) for k in range(3))


@pytest.mark.parametrize("M", [2, 4, 8])
def test_model_acquires_and_tracks(sdr, M):
    """64 channels of M-PSK at offsets 0, +-1e-4 and +-2e-3 turn per symbol with random carrier phases, Es/N0 = 30 dB;
    gains from the loop design with the slope K_d.  After ACQ symbols: RMS phase error modulo 2 pi / M, EVM after a
    real gain fit and |nu 2^-40 - f| within the bars"""
    rng = np.random.default_rng(100 + M)
    offs = [OFFSETS[k % 5] for k in range(64)]
    x, theta, _ = R.psk_rows(M, offs, N, ESN0, rng)
    z, ph, e, nu = R.model(x, design(sdr, M))
    rms, evm, df = R.tracking(M, z, ph, nu, theta, offs, ACQ)
    assert rms.max() < BAR_PHASE and evm.max() < BAR_EVM and df.max() < BAR_FREQ, (rms.max(), evm.max(), df.max())

"""References for the carrier recovery bank (sdr_csync).

Phases are uint64 in units of 2^-64 turn, frequencies int64 in units of 2^-40 turn per symbol, q(x) = rint(x 2^40) for
an f32 x, V = floor(max_freq 2^40).  A loop is (M, kp, ki, err_max, max_freq).  From phi_0, nu_0, for s = 0, 1, ...:
    z_s = x_s r_s,  r_s ~ e^{-2 pi i phi_s / 2^64}
    e_s = 0 for a non-finite g = D_M(z_s), else min(max(g, -err_max), err_max)
    nu_{s+1} = clamp(nu_s + q(fl(ki e_s)), -V, V)
    phi_{s+1} = phi_s + 2^24 (nu_{s+1} + q(fl(kp e_s)))   (mod 2^64)
with D_M GNU Radio's order-M Costas detector (a = sgn(z.re) z.im, b = sgn(z.im) z.re, sgn(-0) = +1, K = f32(sqrt 2 - 1)):
    M = 2: a;  M = 4: fl(a - b);  M = 8: |z.re| >= |z.im| ? fl(a - fl(K b)) : fl(fl(K a) - b)
Everything here is vectorised over channels (rows).  `replay` checks the integer recurrence of reported (phases, errors)
exactly; `model` runs the loop in numpy float32 and exact 64-bit integers with the rotation in f64 (the device rotates
in f32, so the model's z differs from the device's in the last bits and is used for the tracking bars only).
"""
import numpy as np

f32 = np.float32
u64 = np.uint64
TURN_NU = 2.0 ** -40   # one unit of nu, in turns per symbol
TURN_PHI = 2.0 ** -64  # one unit of phi, in turns
K8 = f32(np.sqrt(2.0) - 1.0)


def dev_bound(max_freq):
    """V = floor(max_freq 2^40), exact (scaling a double by 2^40 is exact)"""
    return int(np.floor(float(max_freq) * 2.0 ** 40))


def q(x):
    """rint(x 2^40) of f32 values, exact, as int64"""
    return np.rint(np.asarray(x, f32).astype(np.float64) * 2.0 ** 40).astype(np.int64)


def detector(zr, zi, M):
    """D_M(z) in the dtype of zr, zi (float32: every operation rounded in f32, as the device does)"""
    zr, zi = np.asarray(zr), np.asarray(zi)
    with np.errstate(all="ignore"):
        a = np.where(zr >= 0, zi, -zi)
        b = np.where(zi >= 0, zr, -zr)
        if M == 2:
            return a
        if M == 4:
            return a - b
        K = zr.dtype.type(K8) if zr.dtype == np.float32 else np.sqrt(2.0) - 1.0
        return np.where(np.abs(zr) >= np.abs(zi), a - K * b, K * a - b)


def clamp_err(g, emax):
    """e from g: clamped to [-err_max, err_max], 0 where not finite"""
    g = np.asarray(g, f32)
    with np.errstate(all="ignore"):
        e = np.minimum(np.maximum(g, -f32(emax)), f32(emax))
    return np.where(np.isfinite(g), e, f32(0)).astype(f32)


def slope(M, A=1.0, h=1e-6):
    """K_d: d E[D_M] / d theta at theta = 0 over the constellation at amplitude A, numerically (f64)"""
    pts = A * points(M)

    def d(t):
        z = pts * np.exp(1j * t)
        return detector(z.real, z.imag, M).mean()
    return (d(h) - d(-h)) / (2 * h)


def points(M):
    """the M-PSK constellation of the detector: +-1; (+-1 +- i)/sqrt 2; e^{i pi (2k+1)/8}"""
    if M == 2:
        return np.array([1.0, -1.0], np.complex128)
    return np.exp(1j * np.pi * (2 * np.arange(M) + 1) / M)


def loop_design(bn_t, zeta, kd):
    """(kp, ki) in turns per unit of e: sdr_tsync_loop_design(bn_t, zeta, kd, 1 / (2 pi)) in f64"""
    th = bn_t / (zeta + 1.0 / (4.0 * zeta))
    d = 1.0 + 2.0 * zeta * th + th * th
    return 4.0 * zeta * th / (d * kd) / (2 * np.pi), 4.0 * th * th / (d * kd) / (2 * np.pi)


class Loops:
    """per-channel loop parameters as arrays (a shared loop is repeated)"""

    def __init__(self, loops, C):
        lp = [loops] * C if np.ndim(loops[0]) == 0 else list(loops)
        assert len(lp) == C
        self.M = np.array([int(x[0]) for x in lp])
        self.kp = np.array([x[1] for x in lp], f32)
        self.ki = np.array([x[2] for x in lp], f32)
        self.emax = np.array([x[3] for x in lp], f32)
        self.V = np.array([dev_bound(x[4]) for x in lp], np.int64)

    def err(self, zr, zi):
        """e_s from f32 z for every channel (each with its own order)"""
        g = np.zeros(zr.shape, f32)
        for M in (2, 4, 8):
            m = self.M == M
            if m.any():
                g[m] = detector(zr[m], zi[m], M)
        return clamp_err(g, self.emax)

    def step(self, phi, nu, e, live=None):
        """(phi_{s+1}, nu_{s+1}) from uint64 phi_s, int64 nu_s and f32 e_s; channels not live keep their state"""
        nu1 = np.minimum(np.maximum(nu + q(self.ki * e), -self.V), self.V)
        phi1 = phi + ((nu1 + q(self.kp * e)).astype(u64) << u64(24))
        if live is None:
            return phi1, nu1
        return np.where(live, phi1, phi), np.where(live, nu1, nu)


def replay(phase, err, n, loops, phi0, nu0):
    """asserts every reported phase of C rows (row k: its first n[k] entries) against the recurrence driven by the
    reported errors.  Returns (nu_s [C, max n] int64, (next phi, next nu) per channel)."""
    C = len(n)
    L = Loops(loops, C)
    n = np.asarray(n, np.int64)
    phi = np.array(phi0, u64).reshape(-1) * np.ones(C, u64)
    nu = np.array(nu0, np.int64).reshape(-1) * np.ones(C, np.int64)
    N = int(n.max(initial=0))
    nus = np.zeros((C, N), np.int64)
    for s in range(N):
        live = s < n
        got = np.array([phase[k][s] if live[k] else 0 for k in range(C)], u64)
        bad = live & (got != phi)
        assert not bad.any(), (s, np.nonzero(bad)[0][:4], got[bad][:4], phi[bad][:4])
        nus[:, s] = nu
        e = np.array([err[k][s] if live[k] else 0 for k in range(C)], f32)
        phi, nu = L.step(phi, nu, e, live)
    return nus, (phi, nu)


def rotate(x, phi):
    """x e^{-2 pi i phi / 2^64} in f64 at the exact phases"""
    t = np.asarray(phi, u64).view(np.int64).astype(np.float64) * TURN_PHI
    return np.asarray(x, np.complex128) * np.exp(-2j * np.pi * t)


def model(x, loops, phi0=0, nu0=0):
    """the recurrence over rows x [C, n] with the rotation in f64: (z complex64, phi uint64, e float32, nu int64), each
    [C, n]"""
    x = np.asarray(x, np.complex64)
    C, n = x.shape
    L = Loops(loops, C)
    phi = np.array(phi0, u64).reshape(-1) * np.ones(C, u64)
    nu = np.array(nu0, np.int64).reshape(-1) * np.ones(C, np.int64)
    z = np.empty((C, n), np.complex64)
    ph = np.empty((C, n), u64)
    es = np.empty((C, n), f32)
    nus = np.empty((C, n), np.int64)
    for s in range(n):
        zs = rotate(x[:, s], phi).astype(np.complex64)
        e = L.err(zs.real.astype(f32), zs.imag.astype(f32))
        z[:, s], ph[:, s], es[:, s], nus[:, s] = zs, phi, e, nu
        phi, nu = L.step(phi, nu, e)
    return z, ph, es, nus


def psk_rows(M, offsets, n, esn0_db, rng, A=1.0):
    """C rows of n M-PSK symbols at amplitude A, each rotated by e^{2 pi i (theta_k + f_k s)} with a random carrier
    phase theta_k and the offset f_k (turns per symbol), complex white noise at Es/N0.  Returns (rows complex64,
    theta [C], sent symbols [C, n] complex128)."""
    C = len(offsets)
    pts = points(M)
    a = pts[rng.integers(0, M, (C, n))]
    theta = rng.uniform(0, 1, C)
    s = np.arange(n)
    carrier = np.exp(2j * np.pi * (theta[:, None] + np.asarray(offsets, np.float64)[:, None] * s))
    sigma = A * np.sqrt(10 ** (-esn0_db / 10) / 2)
    w = sigma * (rng.standard_normal((C, n)) + 1j * rng.standard_normal((C, n)))
    return (A * a * carrier + w).astype(np.complex64), theta, a


def tracking(M, z, phase, nu, theta, offsets, skip):
    """per channel, after `skip` symbols: (RMS phase error in radians modulo 2 pi / M against the true carrier, EVM
    against nearest-point decisions after a real gain fit, max |nu 2^-40 - f| in turns per symbol)"""
    C, n = z.shape
    s = np.arange(skip, n)
    t = phase[:, skip:].view(np.int64).astype(np.float64) * TURN_PHI
    d = t - (theta[:, None] + np.asarray(offsets, np.float64)[:, None] * s)
    d = (d + 0.5 / M) % (1.0 / M) - 0.5 / M
    rms = 2 * np.pi * np.sqrt((d ** 2).mean(axis=1))
    y = z[:, skip:].astype(np.complex128)
    pts = points(M)
    dec = pts[np.abs(y[:, :, None] / np.abs(y).mean(axis=1)[:, None, None] - pts).argmin(axis=2)]
    g = (np.conj(y) * dec).real.sum(axis=1) / (np.abs(y) ** 2).sum(axis=1)
    evm = np.sqrt((np.abs(g[:, None] * y - dec) ** 2).mean(axis=1))
    df = np.abs(nu[:, skip:] * TURN_NU - np.asarray(offsets, np.float64)[:, None]).max(axis=1)
    return rms, evm, df

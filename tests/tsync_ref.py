"""References for the symbol timing recovery bank (sdr_tsync).

Positions are Python ints in units of 2^-64 frames (ONE = one frame); loop quantities are ints in units of 2^-40
frames, q(x) = rint(x 2^40) for an f32 x.  Channel k: taps h of length L at P = 2^p times the input rate, nominal
period T, first position tau(0), loop (kp, ki, err_max, max_dev), V = floor(max_dev T) in 2^-40 units.  With v_0 = 0,
y_{-1} = 0, for s = 0, 1, ...:
    T_s = T + 2^24 v_s,  y_s = A(tau_s),  m_s = A(tau_s - floor(T_s / 2))  (s >= 1)
    g = fl(fl(fl(y_s.re - y_{s-1}.re) m_s.re) + fl(fl(y_s.im - y_{s-1}.im) m_s.im))
    e_s = 0 for s = 0 or a non-finite g, else min(max(g, -err_max), err_max)
    v_{s+1} = clamp(v_s - q(fl(ki e_s)), -V, V)
    tau_{s+1} = tau_s + T + 2^24 v_{s+1} - 2^24 q(fl(kp e_s))
A(t) is sdr_arb's interpolant (arb_ref).  Symbol s is released once the frame total n satisfies floor(tau_s) < n.
`model` restates the recurrence with A in f64 (truncated weights) and the loop in numpy float32 and Python ints;
`replay` checks the integer recurrence of reported (positions, errors) exactly.
"""
from fractions import Fraction

import numpy as np

import arb_ref as A

ONE = A.ONE
MASK = A.MASK
f32 = np.float32


def q(x):
    """rint(x 2^40) of an f32 x, exact"""
    return int(np.rint(np.float64(f32(x)) * 2.0 ** 40))


def dev_bound(max_dev, T):
    """V = floor(max_dev T) in units of 2^-40 frames, T in units of 2^-64, from the double's binary value"""
    return (Fraction(float(max_dev)) * int(T)).__floor__() >> 24


def t_min(T, loop):
    """the least step: T - 2^24 V - 2^24 q(fl(kp err_max))"""
    kp, ki, emax, md = loop
    return int(T) - (dev_bound(md, T) << 24) - (q(f32(kp) * f32(emax)) << 24)


def valid(T, loop):
    kp, ki, emax, md = loop
    D = q(f32(kp) * f32(emax)) << 24
    return 2 * D < int(T) - (dev_bound(md, T) << 24)


def max_output(n_in, T, loop):
    """ceil(n_in 2^64 / T_min)"""
    return -(-(int(n_in) * ONE) // t_min(T, loop))


def detector(y, yp, m, emax):
    """e from f32 y_s, y_{s-1}, m_s: every operation rounded in f32, then clamped; 0 when not finite"""
    y, yp, m = np.complex64(y), np.complex64(yp), np.complex64(m)
    with np.errstate(all="ignore"):
        g = (f32(y.real) - f32(yp.real)) * f32(m.real) + (f32(y.imag) - f32(yp.imag)) * f32(m.imag)
    g = f32(g)
    if not np.isfinite(g):
        return f32(0.0)
    return f32(min(max(g, -f32(emax)), f32(emax)))


def loop_step(tau, v, e, T, loop, V):
    """(tau_{s+1}, v_{s+1}) from tau_s, v_s and e_s"""
    kp, ki, emax, md = loop
    v1 = min(max(v - q(f32(ki) * f32(e)), -V), V)
    return tau + int(T) + (v1 << 24) - (q(f32(kp) * f32(e)) << 24), v1


def mid_of(tau, v, T):
    """tau - floor(T_s / 2), T_s = T + 2^24 v"""
    return tau - ((int(T) + (v << 24)) >> 1)


def replay(pos, err, T, loop, first=None, v0=0):
    """positions and period offsets the recurrence gives from the reported errors; asserts every reported position.
    Returns (v_s for every reported symbol, (next tau, next v))."""
    V = dev_bound(loop[3], T)
    tau = int(pos[0]) if first is None else int(first)
    v = v0
    vs = []
    for s in range(len(pos)):
        assert int(pos[s]) == tau, (s, int(pos[s]), tau)
        vs.append(v)
        tau, v = loop_step(tau, v, f32(err[s]), T, loop, V)
    return vs, (tau, v)


class Interp:
    """A(t) of one channel in f64 with the kernel's truncated weights; frames before the row (and past it) are 0"""

    def __init__(self, h, P, y):
        self.h = np.asarray(h, np.float64)
        self.d = np.append(self.h[1:], 0.0) - self.h
        self.P, self.p, self.L = int(P), A.log2(P), self.h.size
        self.y = np.asarray(y, np.complex128)

    def __call__(self, tau):
        n0, f = int(tau) >> 64, int(tau) & MASK
        ip = f >> (64 - self.p) if self.p else 0
        a = (((f << self.p) & MASK) >> 40) * 2.0 ** -24
        j = np.arange(ip, self.L, self.P)
        m = n0 - np.arange(j.size)
        ok = (m >= 0) & (m < self.y.size)
        return complex(((self.h[j] + a * self.d[j]) * np.where(ok, self.y[np.clip(m, 0, self.y.size - 1)], 0)).sum())


def model(h, P, y, T, loop, first=0):
    """the recurrence over one row y (all of it): (y_s complex64, positions, e_s float32, v_s) of the released symbols"""
    A_ = Interp(h, P, y)
    V = dev_bound(loop[3], T)
    n = len(y)
    tau, v, yp = int(first), 0, np.complex64(0)
    ys, pos, es, vs = [], [], [], []
    while (tau >> 64) < n:
        yv = np.complex64(A_(tau))
        e = f32(0.0) if not ys else detector(yv, yp, np.complex64(A_(mid_of(tau, v, T))), loop[2])
        ys.append(yv)
        pos.append(tau)
        es.append(e)
        vs.append(v)
        tau, v = loop_step(tau, v, e, T, loop, V)
        yp = yv
    return np.array(ys, np.complex64), pos, np.array(es, np.float32), vs


def loop_design(bn_t, zeta, ted_gain, period_frames):
    """sdr_tsync_loop_design in f64 (the ABI rounds each gain to f32)"""
    th = bn_t / (zeta + 1.0 / (4.0 * zeta))
    d = 1.0 + 2.0 * zeta * th + th * th
    return 4.0 * zeta * th / (d * ted_gain) * period_frames, 4.0 * th * th / (d * ted_gain) * period_frames


def rrc(u, beta):
    """root-raised-cosine pulse at u symbol periods, unit energy per symbol period"""
    u = np.asarray(u, np.float64)
    out = np.empty_like(u)
    z = np.abs(u) < 1e-9
    s = np.abs(np.abs(4 * beta * u) - 1) < 1e-9
    r = ~(z | s)
    out[z] = 1 - beta + 4 * beta / np.pi
    out[s] = beta / np.sqrt(2) * ((1 + 2 / np.pi) * np.sin(np.pi / (4 * beta)) +
                                  (1 - 2 / np.pi) * np.cos(np.pi / (4 * beta)))
    x = u[r]
    out[r] = (np.sin(np.pi * x * (1 - beta)) + 4 * beta * x * np.cos(np.pi * x * (1 + beta))) / \
        (np.pi * x * (1 - (4 * beta * x) ** 2))
    return out


def rc(u, beta):
    """raised-cosine pulse (the RRC convolved with itself)"""
    u = np.asarray(u, np.float64)
    den = 1 - (2 * beta * u) ** 2
    lim = np.abs(den) < 1e-9
    out = np.sinc(u) * np.cos(np.pi * beta * u) / np.where(lim, 1.0, den)
    return np.where(lim, np.pi / 4 * np.sinc(1 / (2 * beta)), out)


def gardner_slope(beta, span=40):
    """d E[e] / d eps at eps = 0, eps the timing error in symbol periods, for unit-power symbols through RC(beta)"""
    k = np.arange(-span, span + 1, dtype=np.float64)

    def s(eps):
        return ((rc(k + eps, beta) - rc(k - 1 + eps, beta)) * rc(k - 0.5 + eps, beta)).sum()

    h = 1e-4
    return (s(h) - s(-h)) / (2 * h)


def rrc_taps(period, P, beta, span):
    """the matched filter at P times the input rate for a period of `period` frames: L = span period P + 1 taps,
    h[i] = rrc((i / P - c) / period) / period with c the centre, so the output at a symbol's centre is its symbol.
    Returns (taps, c in frames)."""
    L = int(round(span * period * P)) + 1
    c = (L - 1) / (2.0 * P)
    return (rrc((np.arange(L) / P - c) / period, beta) / period).astype(np.float32), c


def qpsk_channel(n_frames, period, delay, beta, span, esn0_db, rng):
    """RRC-shaped QPSK at one symbol per `period` frames (the true period), symbol j centred at delay + j period, unit
    symbol power, complex white noise at Es/N0; returns (row complex64, symbols)"""
    n_sym = int((n_frames - delay) / period) + span + 2
    a = ((rng.integers(0, 2, n_sym) * 2 - 1) + 1j * (rng.integers(0, 2, n_sym) * 2 - 1)) / np.sqrt(2)
    m = np.arange(n_frames, dtype=np.float64)
    x = np.zeros(n_frames, np.complex128)
    j0 = np.floor((m - delay) / period).astype(np.int64)
    for o in range(-span // 2 - 1, span // 2 + 2):
        j = j0 + o
        ok = (j >= 0) & (j < n_sym)
        x += np.where(ok, a[np.clip(j, 0, n_sym - 1)] * rrc((m - delay - j * period) / period, beta), 0)
    sigma2 = period / 10 ** (esn0_db / 10)
    x += np.sqrt(sigma2 / 2) * (rng.standard_normal(n_frames) + 1j * rng.standard_normal(n_frames))
    return x.astype(np.complex64), a


def tracking(pos, ys, vs, T, true_period, delay, centre, skip):
    """after `skip` symbols: (max |timing error| / true period, EVM after a complex gain fit, mean(T + v) / true
    period - 1).  The timing error of tau is its distance to the nearest true centre delay + centre + j true_period."""
    t = np.array([float(Fraction(int(x), ONE)) for x in pos[skip:]])
    ph = (t - delay - centre) / true_period
    err = np.abs(ph - np.round(ph)).max()
    y = np.asarray(ys[skip:], np.complex128)
    dec = (np.sign(y.real) + 1j * np.sign(y.imag)) / np.sqrt(2)
    g = (np.conj(y) * dec).sum() / (np.abs(y) ** 2).sum()
    evm = np.sqrt((np.abs(g * y - dec) ** 2).mean())
    per = np.mean([float(Fraction(int(T) + (int(v) << 24), ONE)) for v in vs[skip:]])
    return err, evm, per / true_period - 1

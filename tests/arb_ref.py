"""References for the arbitrary-ratio resampler bank (sdr_arb).

Positions are Python ints in units of 2^-64 frames (ONE = one frame).  Channel k: taps h of length L at P = 2^p times
the input rate, step sigma, first position tau(0):
    tau(r) = tau(0) + r sigma
    H(t) = (1 - a) h[j] + a h[j+1],  j = floor(t P), a = t P - j,  0 <= j < L (h[L] = 0); 0 otherwise
    z[r] = sum_{0 <= m <= floor(tau(r))} H(tau(r) - m) y[m]
and the computed form: n0 = floor(tau), f its 64-bit fraction, ip = f >> (64 - p), a = ((f << p) mod 2^64) / 2^64
(exact) or ((f << p) mod 2^64 >> 40) 2^-24 (the kernel's truncated weight), c_i = h[iP + ip] + a d[iP + ip] with
d[j] = h[j+1] - h[j], z = sum_{iP + ip < L} c_i y[n0 - i].  After n frames #{r : tau(r) < n} outputs are released.
A row y may start at absolute frame `at`: frame m reads y[m - at] when 0 <= m - at < len(y), else 0.
"""
from fractions import Fraction

import numpy as np

ONE = 1 << 64
MASK = ONE - 1


def log2(P):
    p = int(P).bit_length() - 1
    assert 1 << p == P
    return p


def released(n, first, step):
    """#{r >= 0 : first + r step < n ONE}, exact"""
    x = int(n) * ONE - int(first)
    return 0 if x <= 0 else -(-x // int(step))


def step_of(rate_in, rate_out):
    """sdr_arb_step: rate_in / rate_out to the nearest 2^-64, ties to even; None outside [2^-16, 2^24]"""
    q = round(Fraction(rate_in) / Fraction(rate_out) * ONE)
    return q if (1 << 48) <= q <= (1 << 88) else None


def rrb_first(I, D):
    """(r0, tau(0)) that puts P = I, sigma = D / I on sdr_rrb's outputs r >= r0"""
    r0 = -(-I // D) - 1
    return r0, ((r0 + 1) * D - I) * ONE // I


class Timebase:
    """the piecewise time base of one channel: segments (R_b, tau(R_b), step), one per set_steps"""

    def __init__(self, first, step):
        self.segs = [(0, int(first), int(step))]

    def tau(self, r):
        for rb, base, st in reversed(self.segs):
            if r >= rb:
                return base + (int(r) - rb) * st
        raise ValueError(r)

    def released(self, n):
        x = int(n) * ONE
        for i in range(len(self.segs) - 1, -1, -1):
            rb, base, st = self.segs[i]
            if x > base or i == 0:
                return rb + (0 if x <= base else -(-(x - base) // st))

    def set_step(self, total, step):
        R = self.released(total)
        self.segs.append((R, self.tau(R), int(step)))


def _frame(y, at, m):
    j = m - at
    return y[j] if 0 <= j < len(y) else 0.0


def definition_f64(h, P, y, taus, at=0):
    """the literal definition at the given exact positions: H evaluated at t = tau - m for every m that can contribute"""
    h = np.asarray(h, np.float64)
    L = h.size
    hx = np.append(h, 0.0)
    out = np.zeros(len(taus), np.complex128)
    for o, tau in enumerate(taus):
        n0 = int(tau) >> 64
        acc = 0j
        for m in range(max(0, n0 - L // P - 2), n0 + 1):
            tp = (int(tau) - m * ONE) * P  # t P in units of 2^-64
            j = tp >> 64
            if 0 <= j < L:
                a = (tp & MASK) / ONE
                acc += ((1 - a) * hx[j] + a * hx[j + 1]) * _frame(y, at, m)
        out[o] = acc
    return out


def _split(taus, P):
    p = log2(P)
    n0 = np.array([int(t) >> 64 for t in taus], np.int64)
    f = [int(t) & MASK for t in taus]
    ip = np.array([x >> (64 - p) if p else 0 for x in f], np.int64)
    g = [(x << p) & MASK for x in f]
    return n0, ip, g


def computed_f64(h, P, y, taus, at=0, truncated=False, bound=False):
    """the kernel's chain in f64 at the given exact positions; truncated: the kernel's 2^-24 weights.  bound: also
    return sum |d| |y| per output (the error bound of the weight truncation is 2^-24 times that)"""
    h = np.asarray(h, np.float64)
    y = np.asarray(y, np.complex128)
    L = h.size
    d = np.append(h[1:], 0.0) - h
    n0, ip, g = _split(taus, P)
    if truncated:
        a = np.array([(x >> 40) * 2.0 ** -24 for x in g])
    else:
        a = np.array([x / ONE for x in g])
    T = -(-L // P)
    out = np.zeros(len(taus), np.complex128)
    sad = np.zeros(len(taus))
    step = max(1, (1 << 22) // T)
    for s in range(0, len(taus), step):
        sl = slice(s, s + step)
        i = np.arange(T)
        j = i[None, :] * P + ip[sl, None]
        m = n0[sl, None] - i[None, :] - at
        ok = (j < L) & (m >= 0) & (m < y.size)
        jj = np.minimum(j, L - 1)
        yy = np.where(ok, y[np.clip(m, 0, max(y.size - 1, 0))], 0)
        c = np.where(ok, h[jj] + a[sl, None] * d[jj], 0)
        out[sl] = (c * yy).sum(axis=1)
        sad[sl] = (np.where(ok, np.abs(d[jj]), 0) * np.abs(yy)).sum(axis=1)
    return (out, sad) if bound else out


def terms(P, L, tau):
    """T_ip: the number of terms of the output at tau"""
    ip = _split([tau], P)[1][0]
    return 0 if ip >= L else -(-(L - ip) // P)


def taps_of(h, k):
    h = np.asarray(h)
    return h if h.ndim == 1 else h[k]

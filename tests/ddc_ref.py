"""References for the digital down-converter bank (sdr_ddc).

Channel k: a 64-bit NCO phase phi_k(N) = N inc_k mod 2^64 at absolute stream index N = first_sample + n, the input mixed
down by it, the real low-pass h_k (filter::Fir) and Decimate(D):
    z_k[n] = x[n] e^{-2 pi i phi_k(first + n) / 2^64},   y_k[m] = sum_{j<L} h_k[j] z_k[N_m - j],  N_m = (m + 1) D - 1
and the rotated-taps form the kernels compute,
    y_k[m] = e^{-2 pi i phi_k(first + N_m) / 2^64} sum_j g_k[j] x[N_m - j],  g_k[j] = h_k[j] e^{+2 pi i (j inc_k mod 2^64) / 2^64}.
"""
from fractions import Fraction

import numpy as np

import oracle_lib as O

TWO64 = 1 << 64


def _round_half_away(v):
    """llround / round of C on an exact Fraction"""
    r = (abs(v.numerator) * 2 + v.denominator) // (2 * v.denominator)
    return r if v >= 0 else -r


def phase_increment_exact(freq, rate):
    """sdr_ddc_phase_increment with exact arithmetic: nu = freq / rate (the f64 quotient), nu -= round(nu),
    round(nu 2^64) half away from zero, +-1/2 -> 2^63"""
    nu = Fraction(freq / rate)
    nu -= _round_half_away(nu)
    if abs(nu) == Fraction(1, 2):
        return 1 << 63
    return _round_half_away(nu * TWO64) % TWO64


def rot(phi):
    """e^{-2 pi i phi / 2^64} for uint64 phases (read as signed), f64"""
    turns = np.asarray(phi, np.uint64).astype(np.int64).astype(np.float64) / float(TWO64)
    return np.exp(-2j * np.pi * turns)


def phases(first, idx, inc):
    """(first + idx) * inc mod 2^64, exact"""
    with np.errstate(over="ignore"):
        return (np.uint64(first % TWO64) + np.asarray(idx, np.uint64)) * np.uint64(inc)


def taps_of(h, k):
    h = np.asarray(h, np.float64)
    return h if h.ndim == 1 else h[k]


def rotated_taps(h, inc):
    j = np.arange(len(h), dtype=np.uint64)
    with np.errstate(over="ignore"):
        ph = j * np.uint64(inc)
    return np.asarray(h, np.float64) * np.conj(rot(ph))


def mix_first_f64(h, x, incs, D, first=0):
    """the definition: mix with exact integer phases, filter, decimate: [C, n // D]"""
    x = np.asarray(x, np.complex128)
    n = x.size
    keep = (np.arange(n // D) + 1) * D - 1
    out = np.empty((len(incs), n // D), np.complex128)
    for k, inc in enumerate(incs):
        z = x * rot(phases(first, np.arange(n), inc))
        out[k] = np.convolve(z, taps_of(h, k))[:n][keep]
    return out


def rotated_f64(h, x, incs, D, first=0, outputs=None):
    """the rotated-taps form, optionally only at the given output indices: [C, len(outputs)]"""
    x = np.asarray(x, np.complex128)
    n = x.size
    m = np.arange(n // D) if outputs is None else np.asarray(outputs)
    N = (m + 1) * D - 1
    out = np.empty((len(incs), m.size), np.complex128)
    for k, inc in enumerate(incs):
        g = rotated_taps(taps_of(h, k), inc)
        L = g.size
        idx = N[:, None] - np.arange(L)[None, :]
        xs = np.where(idx >= 0, x[np.clip(idx, 0, n - 1)], 0)
        out[k] = rot(phases(first, N, inc)) * (xs * g[None, :]).sum(axis=1)
    return out


def oracle_f32(h, x, incs, D, first=0):
    """the crate's composition through the CPU oracle: mix in f32 -> Fir(h) -> decimate(D): [C, n // D]"""
    x = np.ascontiguousarray(x, np.complex64)
    rows = []
    for k, inc in enumerate(incs):
        z = (x * rot(phases(first, np.arange(x.size), inc)).astype(np.complex64)).astype(np.complex64)
        y = O.Fir(np.asarray(taps_of(h, k), np.float32)).apply(z)
        rows.append(O.decimate(y, D)[0])
    return np.stack(rows)

"""References for the digital up-converter bank (sdr_duc), the transpose of sdr_ddc.

Channel k (row y_k, frames before the stream 0) is zero-stuffed on sdr_pfs's grid, filtered by its real taps h_k
(Fir<f32, Complex<f32>>), mixed UP by its 64-bit NCO and the channels are summed; F = first_sample is the absolute
index of output 0:
    s_k[(m+1) I - 1] = y_k[m],   u_k[n] = sum_{j<L} h_k[j] s_k[n - j],   x[n] = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64}
and the computed form, n = q I + c - 1:  u_k[n] = sum_i h_k[c + i I] y_k[q - 1 - i].
"""
import numpy as np

import ddc_ref
import oracle_lib as O
import pfs_ref

TWO64 = 1 << 64


def rot_up(phi):
    """e^{+2 pi i phi / 2^64} for uint64 phases, f64"""
    return np.conj(ddc_ref.rot(phi))


def definition_f64(h, y, incs, I, first=0):
    """zero-stuff, np.convolve per channel, the exact integer-phase mixer, the sum: [n I]"""
    y = np.asarray(y, np.complex128)
    n = y.shape[1] * I
    out = np.zeros(n, np.complex128)
    for k, inc in enumerate(incs):
        u = np.convolve(pfs_ref.zero_stuff(y[k], I), ddc_ref.taps_of(h, k))[:n]
        out += u * rot_up(ddc_ref.phases(first, np.arange(n), inc))
    return out


def computed_f64(h, y, incs, I, first=0, outputs=None):
    """the polyphase form the kernel computes, optionally only at the given output indices"""
    y = np.asarray(y, np.complex128)
    nf = y.shape[1]
    n = np.arange(nf * I) if outputs is None else np.asarray(outputs, np.int64)
    c, q = (n + 1) % I, (n + 1) // I
    out = np.zeros(n.size, np.complex128)
    for k, inc in enumerate(incs):
        hk = ddc_ref.taps_of(h, k)
        L = hk.size
        i = np.arange(-(-L // I))
        tap = c[:, None] + i[None, :] * I
        j = q[:, None] - 1 - i[None, :]
        ok = (tap < L) & (j >= 0) & (j < nf)
        u = (np.where(ok, hk[np.minimum(tap, L - 1)], 0) * np.where(ok, y[k][np.clip(j, 0, nf - 1)], 0)).sum(axis=1)
        out += u * rot_up(ddc_ref.phases(first, n, inc))
    return out


def oracle_f32(h, y, incs, I, first=0):
    """the crate's blocks through the CPU oracle: zero-stuff, Fir(h_k) on c64, an f32 mix, the sum in f32"""
    y = np.ascontiguousarray(y, np.complex64)
    n = y.shape[1] * I
    out = np.zeros(n, np.complex64)
    for k, inc in enumerate(incs):
        u = O.Fir(np.asarray(ddc_ref.taps_of(h, k), np.float32)).apply(pfs_ref.zero_stuff(y[k], I))
        out += (u * rot_up(ddc_ref.phases(first, np.arange(n), inc)).astype(np.complex64)).astype(np.complex64)
    return out


def band_limited(n, bw, seed):
    """complex noise whose spectrum is confined to |f| < bw (cycles per sample), unit power, f64"""
    rng = np.random.default_rng(seed)
    spec = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    spec[np.abs(np.fft.fftfreq(n)) >= bw] = 0
    x = np.fft.ifft(spec)
    return x / np.sqrt(np.mean(np.abs(x) ** 2))


def kaiser_pair(D, T, beta=10.0):
    """analysis h (cutoff 0.5/D) and synthesis f = D h, both of length T D + 1: ddc(h) -> duc(f) passes what lies well
    inside each channel with unit gain and a delay of T D samples"""
    h = pfs_ref.kaiser_lowpass(T * D + 1, 0.5 / D, beta)
    return h, D * h

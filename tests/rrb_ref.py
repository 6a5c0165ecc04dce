"""References for the rational resampler bank (sdr_rrb), the textbook upfirdn per channel.

Channel k (row y_k, frames before the stream 0) is zero-stuffed on sdr_pfs's grid, filtered by its real taps h_k
(Fir<f32, Complex<f32>>) and decimated (signal::Decimate keeps sample (r+1) D - 1):
    s_k[(m+1) I - 1] = y_k[m],   u_k[n] = sum_{j<L} h_k[j] s_k[n - j],   z_k[r] = u_k[(r+1) D - 1]
and the computed form, t = (r+1) D - 1, q = (t+1) div I, c = (t+1) mod I:
    z_k[r] = sum_{i < I_c} h_k[c + i I] y_k[q - 1 - i],   I_c = ceil((L - c) / I)
After n frames a channel has released floor(n I / D) outputs.
"""
import numpy as np

import oracle_lib as O
import pfs_ref


def released(n, I, D):
    """outputs after n frames in total, exact (Python integers)"""
    return (int(n) * int(I)) // int(D)


def definition_f64(h, y, I, D):
    """zero-stuff with pfs_ref.zero_stuff, np.convolve, keep (r+1) D - 1: the floor(n I / D) released outputs"""
    y = np.asarray(y, np.complex128)
    u = np.convolve(pfs_ref.zero_stuff(y, I), np.asarray(h, np.float64))[:y.size * I]
    return u[D - 1::D][:released(y.size, I, D)]


def computed_f64(h, y, I, D, outputs=None):
    """the chain the kernel computes, optionally only at the given output indices r"""
    h = np.asarray(h, np.float64)
    y = np.asarray(y, np.complex128)
    L, nf = h.size, y.size
    r = np.arange(released(nf, I, D)) if outputs is None else np.asarray(outputs, np.int64)
    t1 = (r + 1) * D
    q, c = t1 // I, t1 % I
    i = np.arange(-(-L // I))
    tap = c[:, None] + i[None, :] * I
    j = q[:, None] - 1 - i[None, :]
    ok = (tap < L) & (j >= 0) & (j < nf)
    return (np.where(ok, h[np.minimum(tap, L - 1)], 0) * np.where(ok, y[np.clip(j, 0, max(nf - 1, 0))], 0)).sum(axis=1)


def oracle_f32(h, y, I, D):
    """the crate's blocks through the CPU oracle: zero-stuff, Fir(h) on c64, decimate by D"""
    u = O.Fir(np.asarray(h, np.float32)).apply(pfs_ref.zero_stuff(np.asarray(y, np.complex64), I))
    return O.decimate(u, D)[0][:released(len(y), I, D)]


def taps_of(h, k):
    h = np.asarray(h)
    return h if h.ndim == 1 else h[k]

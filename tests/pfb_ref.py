"""References for the polyphase filter bank (sdr_pfb): the definition from the crate's blocks, and its polyphase form.

Channel k of the bank is Fir<Complex<f32>, Complex<f32>> with taps g_k[n] = h[n] e^{+2 pi i k n / M}, followed by
Decimate with wait D: y_k[m] = sum_{n<L} g_k[n] x[(m+1) D - 1 - n], x[<0] = 0 (fir.rs:23-32, adapters/mod.rs:30-37).
"""
import numpy as np

import oracle_lib as O


def modulated_taps(h, M, k):
    n = np.arange(len(h), dtype=np.float64)
    return np.asarray(h, np.float64) * np.exp(2j * np.pi * k * n / M)


def n_frames(n, D):
    return n // D


def direct_f64(h, x, M, D):
    """M modulated FIRs + decimate, in f64 (numpy): [frames, M]"""
    x = np.asarray(x, np.complex128)
    nf = n_frames(x.size, D)
    keep = (np.arange(nf) + 1) * D - 1
    out = np.empty((nf, M), np.complex128)
    for k in range(M):
        out[:, k] = np.convolve(x, modulated_taps(h, M, k))[:x.size][keep]
    return out


def direct_oracle_f32(h, x, M, D):
    """the crate's own blocks through the CPU oracle: Fir(g_k as Complex<f32>) then decimate(D): [frames, M]"""
    x = np.ascontiguousarray(x, np.complex64)
    cols = []
    for k in range(M):
        y = O.Fir(modulated_taps(h, M, k).astype(np.complex64)).apply(x)
        cols.append(O.decimate(y, D)[0])
    return np.stack(cols, axis=1)


def polyphase_f64(h, x, M, D, frames=None, block=None):
    """u_p[m] = sum_t h[tM+p] x[(m+1)D - 1 - tM - p]; v[(-p) mod M] = u_p[m]; y[m] = DFT_M(v) (forward, unnormalised).
    frames: the frame indices to compute (default all).  Returns [len(frames), M]."""
    h = np.asarray(h, np.float64)
    x = np.asarray(x, np.complex128)
    L = h.size
    T = -(-L // M)
    hp = np.zeros(T * M)
    hp[:L] = h
    H = hp.reshape(T, M)                                         # H[t, p] = h[t M + p]
    if frames is None:
        frames = np.arange(n_frames(x.size, D))
    frames = np.asarray(frames, np.int64)
    xp = np.concatenate([np.zeros(T * M, np.complex128), x])     # x[<0] = 0
    off = (np.arange(T)[:, None] * M + np.arange(M)[None, :])    # t M + p
    dst = (-np.arange(M)) % M
    block = block or max(1, (1 << 22) // (T * M))
    out = np.empty((frames.size, M), np.complex128)
    for b0 in range(0, frames.size, block):
        fb = frames[b0:b0 + block]
        e = (fb + 1) * D - 1
        idx = e[:, None, None] - off[None] + T * M
        u = (H[None] * xp[idx]).sum(axis=1)                      # [frames, p]
        v = np.empty_like(u)
        v[:, dst] = u
        out[b0:b0 + block] = np.fft.fft(v, axis=1)
    return out

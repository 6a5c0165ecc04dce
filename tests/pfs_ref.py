"""References for the polyphase synthesis filter bank (sdr_pfs): the definition from the crate's blocks, and its
polyphase form.

Channel k (sample m of frame m) is zero-stuffed by D with sample m at index (m+1) D - 1, filtered by
Fir<Complex<f32>, Complex<f32>> with taps f_k[n] = f[n] e^{+2 pi i k n / M} (fir.rs:23-32), and all channels are summed:
    xh[t] = sum_m sum_k f_k[t - (m+1) D + 1] y_k[m],   0 <= t - (m+1) D + 1 < L
Frame m releases the outputs [m D, (m+1) D), so n frames give n D outputs.
"""
import numpy as np

import oracle_lib as O


def modulated_taps(f, M, k):
    n = np.arange(len(f), dtype=np.float64)
    return np.asarray(f, np.float64) * np.exp(2j * np.pi * k * n / M)


def zero_stuff(col, D):
    """channel samples y[m] placed at (m+1) D - 1 of a stream of len(col) D samples"""
    z = np.zeros(len(col) * D, np.result_type(col, np.complex64))
    z[D - 1::D] = col
    return z


def direct_f64(f, frames, M, D):
    """zero-stuff + M modulated FIRs + sum, in f64 (numpy).  frames: [n, M] -> [n D]"""
    y = np.asarray(frames, np.complex128)
    n = y.shape[0]
    out = np.zeros(n * D, np.complex128)
    for k in range(M):
        out += np.convolve(zero_stuff(y[:, k], D), modulated_taps(f, M, k))[:n * D]
    return out


def direct_oracle_f32(f, frames, M, D):
    """the crate's own blocks through the CPU oracle: zero-stuff, Fir(f_k as Complex<f32>) per channel, summed in f32"""
    y = np.ascontiguousarray(frames, np.complex64)
    out = np.zeros(y.shape[0] * D, np.complex64)
    for k in range(M):
        out += O.Fir(modulated_taps(f, M, k).astype(np.complex64)).apply(zero_stuff(y[:, k], D))
    return out


def polyphase_f64(f, frames, M, D, outputs=None):
    """V_m[r] = Y_m[(-r) mod M] with Y_m = DFT_M(frame m) (forward, unnormalised);
    xh[t] = sum_{n < L, n = t+1 (mod D)} f[n] V_{(t+1-n)/D - 1}[n mod M], frames before the stream zero.
    outputs: the sample indices to compute (default all n D).  Only the frames they need are transformed."""
    f = np.asarray(f, np.float64)
    L = f.size
    n_frames = frames.shape[0]
    t = np.arange(n_frames * D) if outputs is None else np.asarray(outputs, np.int64)
    c, q = (t + 1) % D, (t + 1) // D
    I = -(-L // D)
    i = np.arange(I)
    n = c[:, None] + i[None, :] * D                               # [outputs, I]
    j = q[:, None] - 1 - i[None, :]                               # frame of each tap
    ok = (n < L) & (j >= 0)
    need = np.unique(j[ok])
    Y = np.fft.fft(np.asarray(frames[need], np.complex128), axis=1)
    pos = np.searchsorted(need, np.where(ok, j, need[0] if need.size else 0))
    col = (-(n % M)) % M
    v = np.where(ok, Y[pos, col] if need.size else 0, 0)
    return (np.where(ok, f[np.minimum(n, L - 1)], 0) * v).sum(axis=1)


def kaiser_lowpass(L, cutoff, beta=10.0):
    """Kaiser-windowed sinc of length L, cutoff in cycles per sample, unit DC gain (scipy.signal.firwin's design)"""
    n = np.arange(L) - (L - 1) / 2.0
    h = 2 * cutoff * np.sinc(2 * cutoff * n) * np.kaiser(L, beta)
    return h / h.sum()


def prototype_pair(M, D, T):
    """analysis h (cutoff 0.5/M, a Nyquist(M) filter) and synthesis f (cutoff 1/M, times D), both of length T M + 1:
    Pfb(h) -> Pfs(f) reconstructs x[t - T M] with unit gain"""
    L = T * M + 1
    return kaiser_lowpass(L, 0.5 / M), D * kaiser_lowpass(L, 1.0 / M)

"""References for the averaged power-spectrum estimator (sdr_psd).

Frame j holds the N samples ending at input sample (j + 1) H - 1, x[<0] = 0 (Window + Decimate); X_j = DFT(w * frame_j)
(times 1/sqrt(N) with NORM); spectrum g = mean of |X_j|^2 over frames gK .. gK + K - 1.  SHIFT orders bins as
sdr_fft_labels: slot i holds bin (i - N // 2) mod N.
"""
import numpy as np

S = 32  # frames per chunk of the summation order


def frames(x, N, H, count, first=0):
    """frames first .. first + count - 1 as a [count, N] complex128 array"""
    x = np.asarray(x, np.complex128)
    pad = np.concatenate([np.zeros(N, np.complex128), x])
    out = np.empty((count, N), np.complex128)
    for r in range(count):
        e = (first + r + 1) * H  # one past the frame's last sample
        out[r] = pad[e: e + N]  # pad index e + N - 1 - N = x index e - 1
    return out


def spectra_count(n_samples, H, K):
    return (n_samples // H) // K


def power_f64(x, N, H, K, window=None, shift=True, norm=True):
    """[n_spectra, N] float64: the definition computed with numpy's f64 FFT"""
    G = spectra_count(len(x), H, K)
    if G == 0:
        return np.zeros((0, N))
    w = np.ones(N) if window is None else np.asarray(window, np.float64)
    X = np.fft.fft(frames(x, N, H, G * K) * w, axis=1)
    P = (np.abs(X) ** 2).reshape(G, K, N).mean(axis=1)
    if norm:
        P = P / N
    if shift:
        P = np.roll(P, N // 2, axis=1)
    return P


def power_literal(x, N, H, K, window=None, shift=True, norm=True):
    """the crate chain restated literally: a deque of N samples that starts as N zeros and takes one sample at a time
    (Window), every H-th deque kept (Decimate), a direct DFT sum, |.|^2, the mean of K, the shift of fft.rs"""
    from collections import deque
    w = np.ones(N) if window is None else np.asarray(window, np.float64)
    dq = deque([0j] * N, maxlen=N)
    n = np.arange(N)
    dft = np.exp(-2j * np.pi * np.outer(n, n) / N)
    rows, acc, have = [], np.zeros(N), 0
    for i, s in enumerate(np.asarray(x, np.complex128)):
        dq.append(s)
        if (i + 1) % H:
            continue
        X = dft @ (w * np.array(dq))
        if norm:
            X = X / np.sqrt(N)
        acc = acc + np.abs(X) ** 2
        have += 1
        if have == K:
            P = acc / K
            if shift:
                P = np.array([P[(k - N // 2) % N] for k in range(N)])
            rows.append(P)
            acc, have = np.zeros(N), 0
    return np.array(rows).reshape(len(rows), N)


def chunked(power_rows, K):
    """the library's summation order applied to per-frame |X_j|^2 rows [G K, N] (any float dtype): chunks of S frames
    anchored on each group's first frame, summed in f32 in ascending j, chunk partials summed in f64, times 1/K"""
    p = np.asarray(power_rows, np.float32)
    G = p.shape[0] // K
    out = np.empty((G, p.shape[1]))
    for g in range(G):
        tot = np.zeros(p.shape[1])
        for c0 in range(0, K, S):
            part = np.zeros(p.shape[1], np.float32)
            for j in range(g * K + c0, g * K + min(c0 + S, K)):
                part = part + p[j]
            tot = tot + part.astype(np.float64)
        out[g] = tot * (1.0 / K)
    return out


def bar(N):
    """per-spectrum tolerance relative to the spectrum's max: the FFT bar carried through |.|^2"""
    return 2 * 1e-5 * max(np.log2(N), 1.0)

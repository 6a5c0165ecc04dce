"""References for the fast-convolution synthesis bank (sdr_fcsb), the inverse of sdr_fcfb.

Channel k (row y_k of n_time / I_k frames, frames before the stream 0) is sdr_duc's channel with its own
interpolation I_k: zero-stuffed on sdr_pfs's grid, filtered by h_k, mixed UP by its 64-bit NCO; the channels are
summed.  F = first_sample is the absolute index of output 0:
    s_k[(m+1) I_k - 1] = y_k[m],   u_k[n] = sum_{j<L} h_k[j] s_k[n - j],   x[n] = sum_k u_k[n] e^{+2 pi i phi_k(F + n) / 2^64}
The bank computes it rotate-first by overlap-save on sdr_fcfb's geometry (Il = lcm(I_k), N, P; block b holds the
outputs at absolute indices [b P + eps, (b + 1) P + eps), eps = F mod Il).  `overlap_save_f64` restates the unfold
(frames at span positions g_k u + rho_k, an M_k-point DFT, G'_k[r] = DFT_N(g_k)[r] e^{-2 pi i r rho_k / N}, the sum over
channels and one N-point inverse) in f64 so that the host tests can check it against the definition.
"""
import numpy as np

import ddc_ref as R
import duc_ref
import fcfb_ref
import pfs_ref

TWO64 = 1 << 64
geometry = fcfb_ref.geometry
lcm_of = fcfb_ref.lcm_of
off0 = fcfb_ref.off0


def counts(total, P, o0):
    """outputs released after `total` output positions: those of the completed blocks"""
    return max(0, (total + o0) // P * P - o0)


def n_time_of(rows, Is):
    n = {len(r) * int(i) for r, i in zip(rows, Is)}
    assert len(n) == 1, "n_k I_k must be equal for every channel"
    return n.pop()


def definition_f64(h, rows, incs, Is, first=0):
    """zero-stuff, np.convolve per channel, the exact integer-phase mixer, the sum: [n_time]"""
    n = n_time_of(rows, Is)
    out = np.zeros(n, np.complex128)
    for k, (inc, I) in enumerate(zip(incs, Is)):
        s = pfs_ref.zero_stuff(np.asarray(rows[k], np.complex128), int(I))
        u = np.convolve(s, R.taps_of(h, k))[:n]
        out += u * duc_ref.rot_up(R.phases(first, np.arange(n), inc))
    return out


def overlap_save_f64(h, rows, incs, Is, first=0):
    """the bank's computation in f64 on the absolute block grid: per block and channel the rotated frames at span
    positions g_k u + rho_k, an M_k-point DFT, the unfold with G'_k, the sum over channels, one N-point inverse and the
    last P positions.  Returns the released outputs."""
    n = n_time_of(rows, Is)
    L = np.shape(h)[-1]
    N, P = geometry(L, Is)
    o0 = off0(first, Is, P)
    spec = []
    r = np.arange(N)
    for k, (inc, I) in enumerate(zip(incs, Is)):
        I = int(I)
        g = I & -I
        rho = (N - P - 1) % I
        G = np.fft.fft(np.concatenate([R.rotated_taps(R.taps_of(h, k), inc), np.zeros(N - L)]))
        spec.append((I, g, rho, G * np.exp(-2j * np.pi * ((r * rho) % N) / N)))
    out = []
    for j in range((n + o0) // P):
        s0 = (j + 1) * P - o0 - N
        S = np.zeros(N, np.complex128)
        for k, (I, g, rho, Gp) in enumerate(spec):
            M = N // g
            t = g * np.arange(M) + rho                   # span positions of v
            pos = s0 + t                                 # handle output index
            m = (pos + 1) // I - 1                       # frame index where pos is a frame position
            frame = ((np.arange(M) % (I // g)) == 0) & (t < N) & (m >= 0)
            v = np.zeros(M, np.complex128)
            a = np.array([(first + int(p)) % TWO64 for p in pos[frame]], np.uint64)  # absolute indices
            v[frame] = np.asarray(rows[k], np.complex128)[m[frame]] * duc_ref.rot_up(R.phases(0, a, incs[k]))
            S += Gp * np.fft.fft(v)[r % M]
        x = np.fft.ifft(S)[N - P:]
        nn = j * P - o0 + np.arange(P)
        out.append(x[nn >= 0])
    return np.concatenate(out) if out else np.zeros(0, np.complex128)


def kaiser_pairs(Is, L):
    """duc_ref.kaiser_pair per channel, all of length L (L - 1 a multiple of every I_k): analysis rows h_k (cutoff
    0.5 / I_k) and synthesis rows f_k = I_k h_k; fcfb(h) -> fcsb(f) passes what lies well inside each channel with unit
    gain and a delay of L - 1 samples"""
    pairs = [duc_ref.kaiser_pair(int(I), (L - 1) // int(I)) for I in Is]
    assert all(p[0].size == L for p in pairs)
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])

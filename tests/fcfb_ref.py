"""References for the fast-convolution channel bank (sdr_fcfb).

Channel k is sdr_ddc's channel with its own decimation D_k (ddc_ref's definition per channel).  The bank computes it by
overlap-save on blocks of the absolute stream grid: Dl = lcm(D_k), N = the smallest power of two >= 1024 with
P = floor((N - L + 1) / Dl) Dl >= N / 2; block b holds the outputs at absolute indices [b P + eps, (b + 1) P + eps),
eps = first mod Dl, and is computed from the N inputs ending at its last output.  `overlap_save_f64` restates the
spectral fold and pick in f64 so that the host tests can check it against the definition.
"""
from math import gcd

import numpy as np

import ddc_ref as R

MIN_N, MAX_N = 1024, 1 << 22


def lcm_of(ds):
    out = 1
    for d in ds:
        out = out // gcd(out, int(d)) * int(d)
    return out


def geometry(L, ds):
    """(N, P) of sdr_fcfb_geometry, or None where it returns SDR_ERR_UNSUPPORTED"""
    Dl = lcm_of(ds)
    if Dl > MAX_N:
        return None
    N = MIN_N
    while N <= MAX_N:
        span = N - L + 1
        if span > 0:
            P = span // Dl * Dl
            if P > 0 and 2 * P >= N:
                return N, P
        N *= 2
    return None


def off0(first, ds, P):
    """handle block 0 starts at handle index -off0"""
    eps = first % lcm_of(ds)
    return (first - eps) % P


def counts(total, ds, P, o0):
    """outputs per channel released after `total` inputs: those of the completed blocks"""
    done = max(0, (total + o0) // P * P - o0)
    return [done // int(d) for d in ds]


def definition_f64(h, x, incs, ds, first=0):
    """channel k: mix with exact phases, filter by h_k, decimate by D_k (all outputs of x)"""
    return [R.mix_first_f64(R.taps_of(h, k), x, [inc], int(d), first)[0] for k, (inc, d) in enumerate(zip(incs, ds))]


def overlap_save_f64(h, x, incs, ds, first=0):
    """the bank's computation in f64 on the absolute block grid: per block one N-point DFT, per channel the fold by
    g_k (largest power of two dividing D_k) with G'_k[r] = DFT_N(g_k)[r] e^{+2 pi i r rho_k / N}, an N/g_k-point
    inverse, the pick of every (D_k / g_k)-th and the derotation.  Returns the released outputs per channel."""
    x = np.asarray(x, np.complex128)
    n = x.size
    L = np.shape(h)[-1]
    N, P = geometry(L, ds)
    o0 = off0(first, ds, P)
    nblocks = (n + o0) // P
    spec = []
    for k, (inc, d) in enumerate(zip(incs, ds)):
        d = int(d)
        g = d & -d
        rho = (N - P - 1) % d
        G = np.fft.fft(np.concatenate([R.rotated_taps(R.taps_of(h, k), inc), np.zeros(N - L)]))
        r = np.arange(N)
        spec.append((d, g, rho, G * np.exp(2j * np.pi * ((r * rho) % N) / N)))
    out = [[] for _ in ds]
    for j in range(nblocks):
        s0 = (j + 1) * P - o0 - N
        idx = s0 + np.arange(N)
        span = np.where(idx >= 0, x[np.clip(idx, 0, n - 1)], 0)
        X = np.fft.fft(span)
        for k, (d, g, rho, Gp) in enumerate(spec):
            M = N // g
            F = (Gp * X).reshape(g, M).sum(axis=0)
            c = np.fft.ifft(F) * (M / N)          # (g * x) at span position g u + rho
            i = np.arange(P // d)
            t = N - P + d - 1 + i * d            # kept span positions
            y = c[(t - rho) // g]
            m = (j * P - o0) // d + i
            ok = m >= 0
            a = np.array([(first + s0 + int(v)) % (1 << 64) for v in t[ok]], np.uint64)  # absolute indices
            out[k].append(R.rot(R.phases(0, a, incs[k])) * y[ok])
    return [np.concatenate(o) if o else np.zeros(0, np.complex128) for o in out]

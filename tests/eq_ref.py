"""References for the adaptive equalizer bank (sdr_eq).

One tap count N per bank, 1 <= N <= 64.  Channel k carries weights w[0..N), a delay line x_{s-j} (zeros before the
stream), a symbol total s and an adaptation set (M, mu, a, err_max, S), R = fl(a a).  For each symbol s:
    P_j = w[j] x_{s-j} = (fl(fl(w.re x.re) - fl(w.im x.im)), fl(fl(w.re x.im) + fl(w.im x.re)))
    W   = 2^ceil(log2 min(N, 32)) lanes;  p_l = P_l for l < min(N, W), 0 for N <= l < W;
          N > 32: p_l = fl(P_l + P_{l+32}) where l + 32 < N, else P_l
    y_s = pairwise tree over p_0..p_{W-1}: for o = W/2, ..., 1: p_l <- fl(p_l + p_{l+o});  y_s = p_0
    CMA (s < S): eps = fl(fl(fl(y.re y.re) + fl(y.im y.im)) - R),  g = (fl(eps y.re), fl(eps y.im))
    DD (s >= S): d = D_M(y) at radius a, g = (fl(y.re - d.re), fl(y.im - d.im));  with sgn(-0) = +1:
          M = 2: (+-a, 0);  M = 4: (+-c, +-c), c = f32(a / sqrt 2);
          M = 8: |y.re| >= |y.im| ? (+-p, +-q) : (+-q, +-p), p = f32(a cos pi/8), q = f32(a sin pi/8)
    y or g not finite: e_s = 0 and the taps do not change
    else e_s = each component of g clamped to [-err_max, err_max],  u = (fl(mu e.re), fl(mu e.im))
         w[j] <- (fl(w.re - fl(fl(u.re x.re) + fl(u.im x.im))), fl(w.im - fl(fl(u.im x.re) - fl(u.re x.im))))
`model` restates this in numpy float32 with re and im as separate arrays, so every operation rounds once; it is
vectorised over channels x taps per symbol and reproduces the device's y, e and final taps bit for bit.  Below it: the
multipath workload and the metrics (residual ISI of the combined response, EVM against the sent symbols).
"""
import numpy as np

f32 = np.float32
CMA_ONLY = (1 << 64) - 1
# cos(pi/8) and sin(pi/8) from square roots, which round correctly everywhere (the library uses the same expressions)
COS8 = np.sqrt(2.0 + np.sqrt(2.0)) / 2.0
SIN8 = np.sqrt(2.0 - np.sqrt(2.0)) / 2.0


def lanes(N):
    """W = 2^ceil(log2 min(N, 32))"""
    W = 1
    while W < min(N, 32):
        W *= 2
    return W


def decision_points(M, a):
    """(p, q) of the DD decision at radius a: (+-p, +-q) when |y.re| >= |y.im| (always for M = 2), else (+-q, +-p);
    computed in double and rounded once"""
    a = float(f32(a))
    if M == 2:
        return f32(a), f32(0.0)
    if M == 4:
        c = f32(a / np.sqrt(2.0))
        return c, c
    return f32(a * COS8), f32(a * SIN8)


def centre_spike(N):
    w = np.zeros(N, np.complex64)
    w[(N - 1) // 2] = 1
    return w


class Adapt:
    """per-channel adaptation sets (M, mu, a, err_max, S) as arrays (a shared set is repeated); S = None: CMA only"""

    def __init__(self, adapt, C):
        ad = [adapt] * C if np.ndim(adapt[0]) == 0 else list(adapt)
        assert len(ad) == C
        self.M = np.array([int(a[0]) for a in ad])
        self.mu = np.array([a[1] for a in ad], f32)
        self.a = np.array([a[2] for a in ad], f32)
        self.emax = np.array([a[3] for a in ad], f32)
        self.S = np.array([CMA_ONLY if a[4] is None else int(a[4]) for a in ad], np.uint64)
        self.R = self.a * self.a
        pq = [decision_points(M, a) for M, a in zip(self.M, self.a)]
        self.dp = np.array([p for p, _ in pq], f32)
        self.dq = np.array([q for _, q in pq], f32)
        self.order2 = self.M == 2


def error(yr, yi, s, A):
    """(e.re, e.im, ok) for f32 y of every channel at symbol totals s (uint64 per channel)"""
    with np.errstate(all="ignore"):
        eps = (yr * yr + yi * yi) - A.R
        first = A.order2 | (np.abs(yr) >= np.abs(yi))
        da = np.where(first, A.dp, A.dq)
        db = np.where(first, A.dq, A.dp)
        gdr = yr - np.where(yr >= 0, da, -da)
        gdi = yi - np.where(yi >= 0, db, -db)
        cma = np.asarray(s, np.uint64) < A.S
        gr = np.where(cma, eps * yr, gdr).astype(f32)
        gi = np.where(cma, eps * yi, gdi).astype(f32)
        ok = np.isfinite(yr) & np.isfinite(yi) & np.isfinite(gr) & np.isfinite(gi)
        er = np.where(ok, np.minimum(np.maximum(gr, -A.emax), A.emax), f32(0)).astype(f32)
        ei = np.where(ok, np.minimum(np.maximum(gi, -A.emax), A.emax), f32(0)).astype(f32)
    return er, ei, ok


def taps_rows(taps0, C, N):
    """initial taps [C, N] complex64 from None (centre spike), one row or C rows"""
    if taps0 is None:
        return np.tile(centre_spike(N), (C, 1))
    t = np.asarray(taps0, np.complex64).reshape(-1, N)
    return np.ascontiguousarray(np.broadcast_to(t, (C, N)) if len(t) == 1 else t)


def model(x, N, adapt, taps0=None, n=None):
    """the recurrence over rows x [C, L] (row k's first n[k] symbols, default all) from the creation state.  Returns
    (y, e, taps): y and e complex64 [C, L] (zero past each row's count), taps complex64 [C, N] for the next symbol"""
    x = np.asarray(x, np.complex64)
    C, L = x.shape
    A = Adapt(adapt, C)
    n = np.full(C, L) if n is None else np.asarray(n)
    W = lanes(N)
    m = min(N, W)
    w = taps_rows(taps0, C, N)
    dr, di = np.zeros((C, N), f32), np.zeros((C, N), f32)
    s = np.zeros(C, np.uint64)
    wr, wi = w.real.astype(f32).copy(), w.imag.astype(f32).copy()
    xr, xi = x.real.astype(f32), x.imag.astype(f32)
    y = np.zeros((C, L), np.complex64)
    e = np.zeros((C, L), np.complex64)
    with np.errstate(all="ignore"):
        for t in range(L):
            live = t < n
            dr[live, 1:] = dr[live, :-1]
            di[live, 1:] = di[live, :-1]
            dr[live, 0] = xr[live, t]
            di[live, 0] = xi[live, t]
            Pr = wr * dr - wi * di
            Pi = wr * di + wi * dr
            pr = np.zeros((C, W), f32)
            pi = np.zeros((C, W), f32)
            pr[:, :m] = Pr[:, :m]
            pi[:, :m] = Pi[:, :m]
            if N > 32:
                pr[:, :N - 32] = pr[:, :N - 32] + Pr[:, 32:N]
                pi[:, :N - 32] = pi[:, :N - 32] + Pi[:, 32:N]
            o = W // 2
            while o >= 1:
                pr[:, :o] = pr[:, :o] + pr[:, o:2 * o]
                pi[:, :o] = pi[:, :o] + pi[:, o:2 * o]
                o //= 2
            yr, yi = pr[:, 0], pi[:, 0]
            er, ei, ok = error(yr, yi, s, A)
            y[live, t] = complex_parts(yr, yi)[live]
            e[live, t] = complex_parts(er, ei)[live]
            upd = ok & live
            if upd.any():
                ur = (A.mu * er)[:, None]
                ui = (A.mu * ei)[:, None]
                nwr = wr - (ur * dr + ui * di)
                nwi = wi - (ui * dr - ur * di)
                wr = np.where(upd[:, None], nwr, wr)
                wi = np.where(upd[:, None], nwi, wi)
            s = s + live.astype(np.uint64)
    return y, e, complex_parts(wr, wi)


def complex_parts(re, im):
    """complex64 from separate float32 parts, exactly (signed zeros included)"""
    out = np.empty(np.shape(re), np.complex64)
    out.real = re
    out.imag = im
    return out


# ---- the multipath workload ---------------------------------------------------------------------------------------

def points(M):
    """M-PSK at unit radius: +-1; (+-1 +- i)/sqrt 2; e^{i pi (2k+1)/8}"""
    if M == 2:
        return np.array([1.0, -1.0], np.complex128)
    return np.exp(1j * np.pi * (2 * np.arange(M) + 1) / M)


def multipath_rows(M, C, n, esn0_db, rng, pre=0.25, post=0.4, freq=None):
    """C rows of n symbols of unit-radius M-PSK through a 3-tap symbol-spaced channel per row: a pre-cursor, the main
    tap and a post-cursor, each with a random phase (the main tap's is the carrier phase), normalised to unit energy;
    x_s = h[0] a[s + 2] + h[1] a[s + 1] + h[2] a[s], times e^{2 pi i f s} when freq is given, plus complex white noise
    at Es/N0.  Returns (x complex64 [C, n], h complex128 [C, 3], a complex128 [C, n + 2])."""
    a = points(M)[rng.integers(0, M, (C, n + 2))]
    ph = np.exp(2j * np.pi * rng.uniform(0, 1, (C, 3)))
    h = np.array([pre, 1.0, post])[None, :] * ph
    h /= np.sqrt((np.abs(h) ** 2).sum(axis=1, keepdims=True))
    x = h[:, 0:1] * a[:, 2:] + h[:, 1:2] * a[:, 1:-1] + h[:, 2:3] * a[:, :-2]
    if freq is not None:
        x = x * np.exp(2j * np.pi * np.asarray(freq, np.float64).reshape(-1, 1) * np.arange(n))
    sigma = np.sqrt(10 ** (-esn0_db / 10) / 2)
    x = x + sigma * (rng.standard_normal((C, n)) + 1j * rng.standard_normal((C, n)))
    return x.astype(np.complex64), h, a


def combined(w, h, freq=0.0):
    """c = w * h, the response from sent symbols to y; with a carrier offset f (turns per symbol) tap j of w acts as
    w[j] e^{-2 pi i f j} on the unrotated channel"""
    w = np.asarray(w, np.complex128)
    return np.convolve(w * np.exp(-2j * np.pi * freq * np.arange(len(w))), np.asarray(h, np.complex128))


def isi_db(w, h, freq=0.0):
    """residual ISI of c = w * h in dB: (sum |c|^2 - max |c|^2) / max |c|^2"""
    p = np.abs(combined(w, h, freq)) ** 2
    return 10 * np.log10((p.sum() - p.max()) / p.max())


def evm(y, w, h, a, skip):
    """RMS |y_s / c[delta] - a_{s - delta}| over s >= skip, delta = argmax |c| (a indexed as multipath_rows returns it:
    a_{s - delta} is a[s + 2 - delta])"""
    c = combined(w, h)
    d = int(np.argmax(np.abs(c)))
    s = np.arange(skip, len(y))
    z = np.asarray(y, np.complex128)[skip:] / c[d]
    return float(np.sqrt((np.abs(z - a[s + 2 - d]) ** 2).mean()))

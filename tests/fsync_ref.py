"""References for the frame synchronizer bank (sdr_fsync).

Channel k has a sync word p of Lp c64 values and parameters (F, M, th_search, th_check, V, max_miss, W).  Symbols z_t
are numbered from 0 since create or reset; position s reads z_s .. z_{s+Lp-1}.  Every f32 operation is rounded on its
own, in this order:
    P_j = (fl(fl(p.re z.re) + fl(p.im z.im)), fl(fl(p.re z.im) - fl(p.im z.re)))     (conj(p_j) z_{s+j})
    c_s = P_0, then c_s <- fl(c_s + P_j) for j = 1 .. Lp-1 (componentwise)
    E_s = the same sequential sum of fl(fl(z.re z.re) + fl(z.im z.im)); E_p the same over the word
    a = fl(fl(c.re c.re) + fl(c.im c.im)),  b = fl(E_s E_p),  rho_s = b > 0 ? fl(a / b) : 0
A test passes when rho >= theta (NaN fails).  The best position of the window around e is the s in [e - W, e + W]
with the largest rho (NaN lowest), ties to the smallest |s - e|, then to the earlier s.
State machine (one decision per completed window or searched position, in position order):
    SEARCH from sigma: the first s >= sigma with rho_s >= th_search -> HIT; V = 0: LOCK at once, emit at s, R = r(c_s),
                       e = s + F; else VERIFY with e = s + F, v = 0
    VERIFY: s* = best(e); pass (rho >= th_check): VERIFY_PASS, v += 1, at v = V emit at s* with R = r(c_s*) and LOCK;
            e = s* + F.  Fail: VERIFY_FAIL, SEARCH from e + W + 1
    LOCK:   s* = best(e); pass: LOCK_PASS, R = r(c_s*), m = 0, emit at s*, e = s* + F.  Fail: m += 1; m < max_miss:
            LOCK_MISS, emit at e with R kept, e += F; else LOCK_LOST, SEARCH from e + W + 1
Emitting the frame at s appends D_R(z_t) for t = s + Lp .. s + F - 1 to the channel's payload stream.
`Bank` is the model: numpy float32, vectorised over positions, fed any blocking.
"""
import numpy as np

f32 = np.float32
K8 = f32(np.sqrt(2.0) - 1.0)  # sdr_csync's constant
H8 = f32(1.0 / np.sqrt(2.0))
SEARCH, VERIFY, LOCK = 0, 1, 2
HIT, VERIFY_PASS, VERIFY_FAIL, LOCK_PASS, LOCK_MISS, LOCK_LOST = 1, 2, 3, 4, 5, 6
NO_OUT = (1 << 64) - 1
REC = np.dtype([("pos", "<u8"), ("out_index", "<u8"), ("corr", "<f4", (2,)), ("rho", "<f4"), ("rot", "<u2"),
                ("kind", "<u2")])
assert REC.itemsize == 32


def seq_sum(terms):
    """terms[0] + terms[1] + ... in order, in f32 (terms: [Lp, n])"""
    acc = terms[0].copy()
    for t in terms[1:]:
        acc = acc + t
    return acc


def energy(p):
    """E_p of a word (sequential f32 sum)"""
    p = np.asarray(p, np.complex64)
    return f32(seq_sum([np.atleast_1d(x) for x in (p.real * p.real + p.imag * p.imag)])[0])


def correlate(z, p, Ep):
    """(c, rho) at every position s with s + Lp <= len(z): complex64 and float32 arrays"""
    z = np.asarray(z, np.complex64)
    p = np.asarray(p, np.complex64)
    Lp = len(p)
    n = len(z) - Lp + 1
    if n <= 0:
        return np.zeros(0, np.complex64), np.zeros(0, f32)
    zr, zi = z.real.astype(f32), z.imag.astype(f32)
    pr, pi = p.real.astype(f32), p.imag.astype(f32)
    with np.errstate(all="ignore"):
        cr = pr[0] * zr[:n] + pi[0] * zi[:n]
        ci = pr[0] * zi[:n] - pi[0] * zr[:n]
        es = zr[:n] * zr[:n] + zi[:n] * zi[:n]
        for j in range(1, Lp):
            a, b = zr[j:j + n], zi[j:j + n]
            cr = cr + (pr[j] * a + pi[j] * b)
            ci = ci + (pr[j] * b - pi[j] * a)
            es = es + (a * a + b * b)
        A = cr * cr + ci * ci
        B = es * f32(Ep)
        rho = np.where(B > 0, A / np.where(B > 0, B, f32(1)), f32(0)).astype(f32)
    c = np.empty(n, np.complex64)
    c.real, c.imag = cr, ci
    return c, rho


def rotation(c, M):
    """r(c) in [0, M) of one complex64 value"""
    re, im = f32(np.real(c)), f32(np.imag(c))
    if M == 2:
        return 0 if re >= 0 else 1
    q = (0 if re >= 0 else 2) if abs(re) >= abs(im) else (1 if im >= 0 else 3)
    if M == 4:
        return q
    # c' = c (-i)^q, exact
    for _ in range(q):
        re, im = im, -re
    with np.errstate(all="ignore"):
        t = K8 * re
    o = 1 if im > t else (-1 if im < -t else 0)
    return (2 * q + o) % 8


def derotate(x, r, M):
    """D_r(x) = x e^{-2 pi i r / M} of complex64 values, as the device computes it"""
    x = np.asarray(x, np.complex64)
    re, im = x.real.astype(f32), x.imag.astype(f32)
    if M == 2:
        q = 2 * r
    elif M == 4:
        q = r
    else:
        if r & 1:
            with np.errstate(all="ignore"):
                re, im = (re + im) * H8, (im - re) * H8
        q = r >> 1
    for _ in range(q % 4):
        re, im = im, -re
    out = np.empty(re.shape, np.complex64)
    out.real, out.imag = re, im
    return out


def best(rho, e, W):
    """the best position of the window around e (rho indexed by position)"""
    s = np.arange(e - W, e + W + 1)
    key = rho[s].astype(np.float64)
    key = np.where(np.isnan(key), -1.0, key)
    return int(s[np.lexsort((s, np.abs(s - e), -key))[0]])


class Channel:
    """one channel of the model; feed() takes any blocking and returns (payload, records) of that call"""

    def __init__(self, word, params):
        self.p = np.ascontiguousarray(word, np.complex64)
        self.Lp = len(self.p)
        F, M, ths, thc, V, mm, W = params
        self.F, self.M, self.V, self.mm, self.W = int(F), int(M), int(V), int(mm), int(W)
        self.ths, self.thc = f32(ths), f32(thc)
        self.Ep = energy(self.p)
        self.reset()

    def reset(self):
        self.z = np.zeros(0, np.complex64)
        self.c = np.zeros(0, np.complex64)
        self.rho = np.zeros(0, f32)
        self.state, self.pos, self.cnt, self.R = SEARCH, 0, 0, 0
        self.payload = 0
        self.frame = None  # [next symbol, end] of the frame being emitted

    def _grow(self, x):
        n0 = len(self.c)
        self.z = np.concatenate([self.z, np.asarray(x, np.complex64)])
        c, rho = correlate(self.z[n0:], self.p, self.Ep)
        self.c = np.concatenate([self.c, c])
        self.rho = np.concatenate([self.rho, rho])

    def _rec(self, pos, out, s, kind, rot):
        c = self.c[s]
        return (pos, out, (np.real(c), np.imag(c)), self.rho[s], rot, kind)

    def _emit(self, s):
        self.frame = [s + self.Lp, s + self.F]
        at = self.payload
        self.payload += self.F - self.Lp
        return at

    def feed(self, x):
        self._grow(x)
        total = len(self.z)
        pay, recs = [], []
        while True:
            if self.frame is not None:
                a, b = self.frame[0], min(self.frame[1], total)
                if b > a:
                    pay.append(derotate(self.z[a:b], self.R, self.M))
                    self.frame[0] = b
                if self.frame[0] < self.frame[1]:
                    break
                self.frame = None
            W, F = self.W, self.F
            if self.state == SEARCH:
                avail = len(self.rho)
                seg = self.rho[self.pos:avail] if self.pos < avail else self.rho[:0]
                hits = np.nonzero(seg >= self.ths)[0]
                if len(hits) == 0:
                    self.pos = max(self.pos, avail)
                    break
                s = self.pos + int(hits[0])
                if self.V == 0:
                    self.R = rotation(self.c[s], self.M)
                    recs.append(self._rec(s, self._emit(s), s, HIT, self.R))
                    self.state, self.cnt = LOCK, 0
                else:
                    recs.append(self._rec(s, NO_OUT, s, HIT, rotation(self.c[s], self.M)))
                    self.state, self.cnt = VERIFY, 0
                self.pos = s + F
                continue
            e = self.pos
            if e + W >= len(self.rho):
                break
            s = best(self.rho, e, W)
            ok = self.rho[s] >= self.thc
            r = rotation(self.c[s], self.M)
            if self.state == VERIFY:
                if ok:
                    self.cnt += 1
                    if self.cnt == self.V:
                        self.R = r
                        recs.append(self._rec(s, self._emit(s), s, VERIFY_PASS, r))
                        self.state, self.cnt = LOCK, 0
                    else:
                        recs.append(self._rec(s, NO_OUT, s, VERIFY_PASS, r))
                    self.pos = s + F
                else:
                    recs.append(self._rec(e, NO_OUT, s, VERIFY_FAIL, r))
                    self.state, self.pos, self.cnt = SEARCH, e + W + 1, 0
            elif ok:
                self.R = r
                recs.append(self._rec(s, self._emit(s), s, LOCK_PASS, r))
                self.cnt, self.pos = 0, s + F
            else:
                self.cnt += 1
                if self.cnt < self.mm:
                    recs.append(self._rec(e, self._emit(e), s, LOCK_MISS, self.R))
                    self.pos = e + F
                else:
                    recs.append(self._rec(e, NO_OUT, s, LOCK_LOST, r))
                    self.state, self.pos, self.cnt = SEARCH, e + W + 1, 0
        payload = np.concatenate(pay) if pay else np.zeros(0, np.complex64)
        return payload, np.array(recs, REC)

    def state_tuple(self):
        """(state, v or m, sigma or e, R, symbols consumed, payload total), as sdr_fsync_get_state reports them"""
        return self.state, self.cnt, self.pos, self.R, len(self.z), self.payload


class Bank:
    """C channels; words: [Lp] (shared) or [C, Lp]; params: one tuple or one per channel"""

    def __init__(self, words, params, n_channels=None):
        w = np.asarray(words, np.complex64)
        w = w[None] if w.ndim == 1 else w
        prm = [params] if np.ndim(params[0]) == 0 else list(params)
        C = int(n_channels) if n_channels is not None else max(len(w), len(prm))
        self.ch = [Channel(w[0 if len(w) == 1 else k], prm[0 if len(prm) == 1 else k]) for k in range(C)]

    def feed(self, rows):
        out = [ch.feed(r) for ch, r in zip(self.ch, rows)]
        return [o[0] for o in out], [o[1] for o in out]

    def reset(self):
        for ch in self.ch:
            ch.reset()


def model(rows, words, params):
    """(payload rows, record arrays) of one call over whole rows"""
    return Bank(words, params, len(rows)).feed(rows)


def max_output(n, consumed, Lp, F, W):
    """the header's per-call bounds (payload symbols, records) for n symbols after `consumed`"""
    if n == 0:
        return 0, 0
    mult = 1 if Lp >= W else 2
    carried = min(consumed, Lp + 2 * W - 1)
    G = F - W + 1
    return mult * (n + carried), min(n, 2 * ((n - 1) // G) + 2)


# ---- workloads ------------------------------------------------------------------------------------------------------

def psk(M, n, rng):
    """n unit-modulus M-PSK symbols (complex128): BPSK +-1, QPSK (+-1 +- i)/sqrt 2, 8PSK e^{i pi (2k+1)/8}"""
    k = rng.integers(0, M, n)
    if M == 2:
        return (1 - 2 * k).astype(np.complex128)
    return np.exp(1j * np.pi * (2 * k + 1) / M) if M == 8 else np.exp(1j * np.pi * (2 * k + 1) / 4)


def framed(word, F, n_frames, M, rng, rot=0, esn0_db=None, start=0):
    """a stream of `start` random symbols then n_frames frames (the word, then F - Lp random M-PSK symbols), rotated by
    e^{2 pi i rot / M} (rot: one value, or one per frame) with complex Gaussian noise at Es/N0 (None: none).  Returns
    (complex64 stream, complex128 payload symbols per frame before rotation)"""
    word = np.asarray(word, np.complex128)
    Lp = len(word)
    rots = np.broadcast_to(np.asarray(rot), (n_frames,))
    parts, pays = [psk(M, start, rng) * np.exp(2j * np.pi * rots[0] / M)], []
    for j in range(n_frames):
        pay = psk(M, F - Lp, rng)
        pays.append(pay)
        parts.append(np.concatenate([word, pay]) * np.exp(2j * np.pi * rots[j] / M))
    x = np.concatenate(parts)
    if esn0_db is not None:
        s = np.sqrt(10 ** (-esn0_db / 10) / 2)
        x = x + s * (rng.standard_normal(len(x)) + 1j * rng.standard_normal(len(x)))
    return x.astype(np.complex64), pays


def word(Lp, rng, M=4):
    """a random QPSK (or M-PSK) sync word"""
    return psk(M, Lp, rng).astype(np.complex64)

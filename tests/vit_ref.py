"""References for the Viterbi decoder bank (sdr_vit).

Code: constraint length K (3 <= K <= 9), S = 2^(K-1) states, rate 1/n (2 <= n <= 4), generators g_0 .. g_{n-1} in
[1, 2^K) in the usual octal convention, the MSB tapping the current input (802.11: K = 7, (0o133, 0o171)).
Encoder: the state s_{t-1} holds the K - 1 previous inputs, u_{t-1} at bit K - 2;
    r_t = (u_t << (K-1)) | s_{t-1},  c_{t,j} = popcount(r_t & g_j) mod 2,  s_t = r_t >> 1.
Soft input: step t reads n f32 values x[t n + j]; a positive value favours bit 0 (BPSK 0 -> +1).  With the scale
sigma_k of channel k: a non-finite x gives q = 0 (an erasure), else q = rint(clamp(fl(x sigma_k), -127, 127)), half to
even (a product that overflows saturates).
Branch cost: sum_j (c_j ? 127 + q_j : 127 - q_j), an integer in [0, 254 n].
Add-compare-select: the new state s' has predecessors p_b = ((s' << 1) & (S-1)) | b; m'(s') = min_b m(p_b) + cost,
the decision d = 1 only when the b = 1 sum is strictly smaller (ties take b = 0).
Start: zero start m(0) = 0, every other state I = (K-1) 254 n + 1; uniform start: every state 0.
Release: L a multiple of 32, 32 <= L <= 512.  At every per-channel step total T = 32 j with T >= L + 32: the best state
after step T - 1 (least metric, ties to the lowest index), a traceback through steps T-1 .. T-L-32 (step i's bit is
s >> (K-2), the previous state ((s << 1) & (S-1)) | d_i(s)), and the bits of steps [T-L-32, T-L) are released.  After
T steps E(T) = max(0, 32 floor(T/32) - L) bits are out.
Finish: the T - E(T) remaining bits by one traceback from state 0 (terminated) or from the best state; the channel
returns to its creation state.
Metrics are exact int64 and never renormalised: the device may hold them in any width because the spread
max m - min m never exceeds I + (K-2) 254 n (DESIGN K18).
"""
import numpy as np

CODES = {  # name -> (K, generators)
    "gsm": (5, (0o23, 0o33)),
    "k7": (7, (0o133, 0o171)),
    "k7n3": (7, (0o133, 0o171, 0o165)),
    "k9": (9, (0o561, 0o753)),
    "k9n3": (9, (0o557, 0o663, 0o711)),
}


def released(T, L):
    """E(T): bits out after T steps"""
    T = np.asarray(T, np.int64)
    return np.maximum(0, 32 * (T // 32) - L)


def spread_bound(K, n):
    return (2 * K - 3) * 254 * n + 1


def parity(v):
    v = np.asarray(v, np.int64).copy()
    p = np.zeros_like(v)
    while (v != 0).any():
        p ^= v & 1
        v >>= 1
    return p


def encode(bits, K, gens, state=0):
    """bits [C, m] (or [m]) -> code bits [C, m, n] (uint8), from the encoder state `state`"""
    b = np.atleast_2d(np.asarray(bits, np.int64))
    C_, m = b.shape
    s = np.broadcast_to(np.asarray(state, np.int64), (C_,)).copy()
    out = np.empty((C_, m, len(gens)), np.uint8)
    for t in range(m):
        r = (b[:, t] << (K - 1)) | s
        for j, g in enumerate(gens):
            out[:, t, j] = parity(r & g)
        s = r >> 1
    return out if np.ndim(bits) > 1 else out[0]


def quantise(x, scale):
    """q of f32 soft values x [C, ...] at scales sigma [C] (or one): int64"""
    x = np.asarray(x, np.float32)
    s = np.asarray(scale, np.float32).reshape((-1,) + (1,) * (x.ndim - 1))
    with np.errstate(all="ignore"):
        v = x * s
    q = np.rint(np.clip(v, np.float32(-127), np.float32(127)))
    q[~np.isfinite(x)] = 0
    return q.astype(np.int64)


def trellis(K, gens):
    """for every new state s' and b: the predecessor p_b and the code pattern sum_j c_j 2^j of that branch"""
    S = 1 << (K - 1)
    sp = np.arange(S, dtype=np.int64)
    pred = np.stack([((sp << 1) & (S - 1)) | b for b in (0, 1)])                        # [2, S]
    r = ((sp >> (K - 2)) << (K - 1))[None] | pred
    pat = sum(parity(r & g) << j for j, g in enumerate(gens))                             # [2, S]
    return pred, pat


class Vit:
    """the bank's definition for C channels, streaming: process() and finish() release exactly the device's bits"""

    def __init__(self, K, gens, L, scale, zero_start, C=None):
        self.K, self.gens, self.L, self.n = int(K), tuple(int(g) for g in gens), int(L), len(gens)
        sc = np.atleast_1d(np.asarray(scale, np.float32))
        self.C = int(C) if C is not None else len(sc)
        self.scale = np.broadcast_to(sc, (self.C,)).copy()
        self.zero_start = bool(zero_start)
        self.S = 1 << (self.K - 1)
        self.R = self.L + 32
        self.pred, self.pat = trellis(self.K, self.gens)
        P = 1 << self.n
        self.sgn = np.array([[1 if (p >> j) & 1 else -1 for j in range(self.n)] for p in range(P)], np.int64)
        self.I = (self.K - 1) * 254 * self.n + 1
        self.m = np.zeros((self.C, self.S), np.int64)
        self.dec = np.zeros((self.C, self.R, self.S), np.uint8)
        self.T = np.zeros(self.C, np.int64)
        for k in range(self.C):
            self._init(k)

    def _init(self, k):
        self.m[k] = 0
        if self.zero_start:
            self.m[k, 1:] = self.I
        self.T[k] = 0

    def _trace(self, ks, s, top, count):
        """from states s after step top - 1 of channels ks: the bits of steps [top - count, top), [len(ks), count]"""
        bits = np.zeros((len(ks), count), np.uint8)
        s = s.astype(np.int64).copy()
        for j in range(count):
            i = top - 1 - j
            bits[:, count - 1 - j] = s >> (self.K - 2)
            d = self.dec[ks, i % self.R, s]
            s = ((s << 1) & (self.S - 1)) | d
        return bits

    def process(self, x, n=None):
        """x: [C, steps, n] or [C, steps * n] f32; n: steps per channel (default all) -> C uint8 arrays of released
        bits"""
        x = np.asarray(x, np.float32).reshape(self.C, -1, self.n)
        steps = np.full(self.C, x.shape[1], np.int64) if n is None else np.asarray(n, np.int64).reshape(self.C)
        q = quantise(x, self.scale)                                                       # [C, steps, n]
        base = 127 * self.n
        out = [[] for _ in range(self.C)]
        p0, p1 = self.pred
        c0, c1 = self.pat
        for t in range(int(steps.max()) if self.C else 0):
            act = np.nonzero(t < steps)[0]
            cost = base + q[act, t] @ self.sgn.T                                          # [A, P]
            m = self.m[act]
            a0 = m[:, p0] + cost[:, c0]
            a1 = m[:, p1] + cost[:, c1]
            d = a1 < a0
            self.m[act] = np.where(d, a1, a0)
            self.dec[act, self.T[act] % self.R] = d
            self.T[act] += 1
            T = self.T[act]
            rel = act[(T % 32 == 0) & (T >= self.L + 32)]
            if len(rel):
                top = int(self.T[rel[0]])
                same = self.T[rel] == top
                for grp in ([rel] if same.all() else [[k] for k in rel]):
                    grp = np.asarray(grp)
                    top = int(self.T[grp[0]])
                    best = np.argmin(self.m[grp], axis=1)
                    b = self._trace(grp, best, top, self.L + 32)[:, :32]
                    for i, k in enumerate(grp):
                        out[k].append(b[i])
        return [np.concatenate(o) if o else np.zeros(0, np.uint8) for o in out]

    def finish(self, which=None, terminated=True):
        """the remaining T - E(T) bits of the channels in `which` (None: all); they return to the creation state"""
        sel = np.ones(self.C, bool) if which is None else np.asarray(which, bool).reshape(self.C)
        out = [np.zeros(0, np.uint8) for _ in range(self.C)]
        for k in np.nonzero(sel)[0]:
            T = int(self.T[k])
            cnt = T - int(released(T, self.L))
            if cnt:
                s = np.array([0 if terminated else int(np.argmin(self.m[k]))])
                out[k] = self._trace(np.array([k]), s, T, cnt)[0]
            self._init(k)
        return out

    def output_count(self, n_in):
        n_in = np.asarray(n_in, np.int64)
        return released(self.T + n_in, self.L) - released(self.T, self.L)


def model(x, K, gens, L, scale, zero_start, n=None):
    """the released bits of a fresh bank fed x ([C, steps, n] or [C, steps * n] f32) in one call: C uint8 arrays"""
    x = np.asarray(x, np.float32)
    return Vit(K, gens, L, scale, zero_start, C=x.shape[0]).process(x, n)


def finish(v, which=None, terminated=True):
    return v.finish(which, terminated)


def bpsk(code_bits, ebn0_db, rate, rng, amp=1.0):
    """code bits -> f32 soft values amp (1 - 2c) + noise at Eb/N0 (dB) for a code of rate `rate`"""
    sigma = np.sqrt(1.0 / (2.0 * rate * 10.0 ** (ebn0_db / 10.0)))
    c = np.asarray(code_bits, np.float64)
    return (amp * ((1.0 - 2.0 * c) + sigma * rng.standard_normal(c.shape))).astype(np.float32)

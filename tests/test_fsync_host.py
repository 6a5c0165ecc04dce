"""CPU: the frame synchronizer bank's reference model (fsync_ref) and ABI without a device.  create rejects every
invalid parameter and fails with NO_DEVICE for a valid one; NULL handles give NULL_HANDLE.  The vectorised model equals
a scalar restatement fed one symbol at a time on streams that reach every transition and record kind; r(c) and D_r
hold at every sector edge; max_output's bounds are never exceeded, under any blocking, on streams built to maximise
records and payload; the model's outputs do not depend on the blocking; and the detection statistics that set the GPU
bars (false hits on 10^7 random QPSK positions at Lp = 64, acquisition and lock hold at a few Es/N0)."""
import ctypes as C

import numpy as np
import pytest

import fsync_ref as R

F32 = np.float32


# ---- ABI without a device -------------------------------------------------------------------------------------------

def _cfg(sdr, Lp, words, params, C_, n_words=None, n_params=None):
    """the config keeps its arrays alive"""
    w = None if words is None else np.ascontiguousarray(words, np.complex64)
    P = None if params is None else (sdr._ffi.FsyncParams * len(params))(*[sdr._ffi.FsyncParams(*p) for p in params])
    cfg = sdr._ffi.FsyncConfig(Lp, None if w is None else w.ctypes.data,
                               (0 if w is None else len(w)) if n_words is None else n_words,
                               None if P is None else C.addressof(P),
                               (0 if P is None else len(params)) if n_params is None else n_params, C_, 0, None)
    cfg.keep = (w, P)
    return cfg


def test_fsync_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    rng = np.random.default_rng(0)
    w16 = R.word(16, rng)[None]
    ok = (100, 4, 0.5, 0.3, 2, 3, 4)
    bad_params = [(100, 3, 0.5, 0.3, 2, 3, 4), (100, 16, 0.5, 0.3, 2, 3, 4), (100, 0, 0.5, 0.3, 2, 3, 4),
                  (100, 4, 0.0, 0.3, 2, 3, 4), (100, 4, 1.0001, 0.3, 2, 3, 4), (100, 4, float("nan"), 0.3, 2, 3, 4),
                  (100, 4, -0.5, 0.3, 2, 3, 4), (100, 4, 0.5, 0.0, 2, 3, 4), (100, 4, 0.5, 1.5, 2, 3, 4),
                  (100, 4, 0.5, float("nan"), 2, 3, 4), (100, 4, 0.5, 0.3, 9, 3, 4), (100, 4, 0.5, 0.3, 2, 0, 4),
                  (100, 4, 0.5, 0.3, 2, 256, 4), (100, 4, 0.5, 0.3, 2, 3, 33),
                  (24, 4, 0.5, 0.3, 2, 3, 4),                # F = Lp + 2W
                  (16, 4, 0.5, 0.3, 2, 3, 0),                # F = Lp
                  ((1 << 24) + 1, 4, 0.5, 0.3, 2, 3, 4)]     # F > 2^24
    assert lib.sdr_fsync_create(None, C.byref(err)) is None and err.value == 100
    nanw = w16.copy()
    nanw[0, 3] = np.nan
    infw = w16.copy()
    infw[0, 5] = np.inf + 0j
    big = np.full((1, 16), 1e20 + 0j, np.complex64)   # E_p overflows
    bad = [_cfg(sdr, 16, None, [ok], 4, n_words=1),                        # NULL words
           _cfg(sdr, 16, w16, None, 4, n_params=1),                        # NULL params
           _cfg(sdr, 7, w16[:, :7], [ok], 4),                              # Lp < 8
           _cfg(sdr, 1025, np.ones((1, 1025)), [(2000, 4, 0.5, 0.3, 2, 3, 4)], 4),  # Lp > 1024
           _cfg(sdr, 16, np.concatenate([w16, w16]), [ok], 4),             # n_words not in {1, C}
           _cfg(sdr, 16, w16, [ok, ok], 4),                                # n_params not in {1, C}
           _cfg(sdr, 16, w16, [ok], 0),                                    # C = 0
           _cfg(sdr, 16, w16, [ok], 65537),                                # C > 65536
           _cfg(sdr, 16, nanw, [ok], 4), _cfg(sdr, 16, infw, [ok], 4),     # non-finite words
           _cfg(sdr, 16, np.zeros((1, 16)), [ok], 4),                      # E_p = 0
           _cfg(sdr, 16, big, [ok], 4)]                                    # E_p not finite
    bad += [_cfg(sdr, 16, w16, [ok] * 3 + [p], 4) for p in bad_params]
    for i, cfg in enumerate(bad):
        err.value = 0
        assert lib.sdr_fsync_create(C.byref(cfg), C.byref(err)) is None and err.value == 100, i
    n = np.zeros(4, np.uintp)
    st = sdr._ffi.FsyncState()
    assert lib.sdr_fsync_process(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data, None, 0, 0, None) == 103
    assert lib.sdr_fsync_process_dev(None, None, n.ctypes.data, 0, None, 0, 0, n.ctypes.data, None, 0, 0, None) == 103
    assert lib.sdr_fsync_max_output(None, n.ctypes.data, n.ctypes.data, n.ctypes.data) == 103
    assert lib.sdr_fsync_get_state(None, 0, C.byref(st)) == 103
    assert lib.sdr_fsync_reset(None) == 103
    assert lib.sdr_fsync_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_fsync_destroy(None)
    if sdr.device_count() == 0:
        # valid, at the edges: Lp 8 and 1024, F = Lp + 2W + 1 and 2^24, every order, V 0 and 8, max_miss 1 and 255,
        # W 0 and 32, thresholds 1, per-channel words and params, C = 65536
        edge = [(8 + 64 + 1, 2, 1.0, 1.0, 0, 1, 32), (1 << 24, 4, 1e-6, 1e-6, 8, 255, 0), (9, 8, 0.5, 0.5, 3, 2, 0),
                (100, 4, 0.5, 0.3, 2, 3, 4)]
        for cfg in [_cfg(sdr, 8, R.word(8, rng)[None].repeat(4, 0), edge, 4), _cfg(sdr, 16, w16, [ok], 65536),
                    _cfg(sdr, 1024, R.word(1024, rng)[None], [(1024 + 65, 8, 0.5, 0.3, 1, 1, 32)], 3)]:
            err.value = 0
            assert lib.sdr_fsync_create(C.byref(cfg), C.byref(err)) is None and err.value == 102


def test_fsync_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Fsync(R.word(32, np.random.default_rng(1)), (200, 4, 0.5, 0.3, 1, 2, 2), n_channels=3)
    assert e.value.code == 102


# ---- rotation and derotation ----------------------------------------------------------------------------------------

def _signed(re, im):
    a = np.zeros(1, np.complex64)
    a.real[0], a.imag[0] = F32(re), F32(im)
    return a[0]


def test_rotation_at_sector_edges():
    c = _signed
    K = R.K8
    up = np.nextafter(K, F32(2))
    dn = np.nextafter(K, F32(0))
    tiny = np.float32(1e-45)
    cases = {2: [(c(0.0, 5), 0), (c(-0.0, 5), 0), (c(-0.0, -0.0), 0), (c(-tiny, 0), 1), (c(tiny, -3), 0),
                 (c(np.nan, 1), 1)],
             4: [(c(1, 1), 0), (c(-1, 1), 2), (c(1, -1), 0), (c(-1, -1), 2), (c(0, 1), 1), (c(0, -1), 3),
                 (c(-0.0, -0.0), 0), (c(0.0, -0.0), 0), (c(-0.0, 0.0), 0), (c(np.nextafter(F32(1), F32(0)), 1), 1),
                 (c(-np.nextafter(F32(1), F32(0)), -1), 3), (c(np.nan, 0), 1), (c(1, np.nan), 3)],
             8: [(c(1, K), 0), (c(1, up), 1), (c(1, -K), 0), (c(1, -up), 7), (c(1, dn), 0), (c(1, 1), 1),
                 (c(1, -1), 7), (c(-K, 1), 2), (c(-up, 1), 3), (c(K, 1), 2), (c(up, 1), 1), (c(-1, K), 4),
                 (c(-1, -K), 4), (c(-1, -up), 5), (c(K, -1), 6), (c(-up, -1), 5), (c(up, -1), 7),
                 (c(-0.0, -0.0), 0), (c(0.0, -0.0), 0), (c(np.nan, np.nan), 6)]}
    for M, cs in cases.items():
        for i, (v, want) in enumerate(cs):
            assert R.rotation(v, M) == want, (M, i, v)
    # away from the edges r is the nearest multiple of 2 pi / M
    rng = np.random.default_rng(2)
    for M in (2, 4, 8):
        a = rng.uniform(0, 2 * np.pi, 4000)
        frac = a * M / (2 * np.pi)
        keep = np.abs(frac - np.round(frac)) < 0.49
        for ang, f in zip(a[keep], frac[keep]):
            v = np.complex64(rng.uniform(0.1, 100) * np.exp(1j * ang))
            assert R.rotation(v, M) == int(np.round(f)) % M


def test_derotation_exact_and_accurate():
    rng = np.random.default_rng(3)
    x = (rng.standard_normal(1000) + 1j * rng.standard_normal(1000)).astype(np.complex64)
    x[:4] = [0, -0.0, complex(-0.0, -0.0), complex(np.inf, 1)]
    for M in (2, 4):
        for r in range(M):
            d = R.derotate(x, r, M)
            with np.errstate(invalid="ignore"):
                w = x.astype(np.complex128) * np.exp(-2j * np.pi * r / M)
            fin = np.isfinite(x)
            # exact: each component is +-x.re or +-x.im
            assert np.array_equal(np.abs(d.real[fin]) + np.abs(d.imag[fin]), np.abs(x.real[fin]) + np.abs(x.imag[fin]))
            assert np.allclose(d[fin], w[fin], rtol=0, atol=1e-6)
    for r in range(8):
        d = R.derotate(x[4:], r, 8)
        w = x[4:].astype(np.complex128) * np.exp(-2j * np.pi * r / 8)
        assert np.abs(d - w).max() < 4e-7 * np.abs(x[4:]).max()
    # D_{r(c)} brings c into |arg| <= pi / M
    for M in (2, 4, 8):
        c = (rng.standard_normal(500) + 1j * rng.standard_normal(500)).astype(np.complex64)
        for v in c:
            d = R.derotate(np.array([v]), R.rotation(v, M), M)[0]
            assert abs(np.angle(d)) <= np.pi / M + 1e-6


# ---- the model against a scalar restatement -------------------------------------------------------------------------

class Scalar:
    """the definition restated one symbol at a time with scalar f32 arithmetic"""

    def __init__(self, word, prm):
        self.p = [np.complex64(v) for v in word]
        self.Lp = len(word)
        self.F, self.M, ths, thc, self.V, self.mm, self.W = prm
        self.ths, self.thc = F32(ths), F32(thc)
        e = None
        for v in self.p:
            t = F32(v.real) * F32(v.real) + F32(v.imag) * F32(v.imag)
            e = t if e is None else e + t
        self.Ep = e
        self.z, self.c, self.rho = [], [], []
        self.state, self.pos, self.cnt, self.R, self.payload = R.SEARCH, 0, 0, 0, 0
        self.frame = None
        self.out, self.recs = [], []

    def _corr(self, s):
        cr = ci = es = None
        with np.errstate(all="ignore"):
            for j in range(self.Lp):
                p, z = self.p[j], self.z[s + j]
                pr, pi, zr, zi = F32(p.real), F32(p.imag), F32(z.real), F32(z.imag)
                a, b, e = pr * zr + pi * zi, pr * zi - pi * zr, zr * zr + zi * zi
                cr, ci, es = (a, b, e) if j == 0 else (cr + a, ci + b, es + e)
            A, B = cr * cr + ci * ci, es * self.Ep
            rho = A / B if B > 0 else F32(0)
        self.c.append(_signed(cr, ci))
        self.rho.append(F32(rho))

    def _emit(self, s):
        self.frame = [s + self.Lp, s + self.F]
        at = self.payload
        self.payload += self.F - self.Lp
        t = len(self.z)
        while self.frame[0] < min(t, self.frame[1]):
            self.out.append(R.derotate(np.array([self.z[self.frame[0]]]), self.R, self.M)[0])
            self.frame[0] += 1
        return at

    def _best(self, e):
        best = None
        for s in range(e - self.W, e + self.W + 1):
            k = -1.0 if np.isnan(self.rho[s]) else float(self.rho[s])
            key = (k, -abs(s - e), -s)
            if best is None or key > best[0]:
                best = (key, s)
        return best[1]

    def push(self, x):
        self.z.append(np.complex64(x))
        t = len(self.z) - 1
        if self.frame is not None and self.frame[0] == t < self.frame[1]:
            self.out.append(R.derotate(np.array([self.z[t]]), self.R, self.M)[0])
            self.frame[0] += 1
        if t >= self.Lp - 1:
            self._corr(t - self.Lp + 1)
        while True:
            rec = lambda pos, oi, s, kind, rot: self.recs.append((pos, oi, (self.c[s].real, self.c[s].imag),
                                                                  self.rho[s], rot, kind))
            if self.state == R.SEARCH:
                s = t - self.Lp + 1
                if s < self.pos or s < 0 or not self.rho[s] >= self.ths:
                    return
                r = R.rotation(self.c[s], self.M)
                if self.V == 0:
                    self.R = r
                    rec(s, self._emit(s), s, R.HIT, r)
                    self.state = R.LOCK
                else:
                    rec(s, R.NO_OUT, s, R.HIT, r)
                    self.state = R.VERIFY
                self.cnt, self.pos = 0, s + self.F
                continue
            e = self.pos
            if t != e + self.W + self.Lp - 1:
                return
            s = self._best(e)
            ok = self.rho[s] >= self.thc
            r = R.rotation(self.c[s], self.M)
            if self.state == R.VERIFY:
                if ok:
                    self.cnt += 1
                    if self.cnt == self.V:
                        self.R = r
                        rec(s, self._emit(s), s, R.VERIFY_PASS, r)
                        self.state, self.cnt = R.LOCK, 0
                    else:
                        rec(s, R.NO_OUT, s, R.VERIFY_PASS, r)
                    self.pos = s + self.F
                else:
                    rec(e, R.NO_OUT, s, R.VERIFY_FAIL, r)
                    self.state, self.pos, self.cnt = R.SEARCH, e + self.W + 1, 0
            elif ok:
                self.R = r
                rec(s, self._emit(s), s, R.LOCK_PASS, r)
                self.cnt, self.pos = 0, s + self.F
            else:
                self.cnt += 1
                if self.cnt < self.mm:
                    rec(e, self._emit(e), s, R.LOCK_MISS, self.R)
                    self.pos = e + self.F
                else:
                    rec(e, R.NO_OUT, s, R.LOCK_LOST, r)
                    self.state, self.pos, self.cnt = R.SEARCH, e + self.W + 1, 0


def eventful(word, F, M, n_frames, rng, W=2, special=True):
    """frames with rotations changing every few frames, a deleted and an inserted symbol, frames whose word is missing,
    a false word between frames, noise, and (special) NaN, Inf, zero and overflowing stretches"""
    Lp = len(word)
    rots = np.repeat(rng.integers(0, M, n_frames // 3 + 1), 3)[:n_frames]
    x, _ = R.framed(word, F, n_frames, M, rng, rots, esn0_db=12.0, start=int(rng.integers(0, F)))
    x = list(x)
    start = len(x) - n_frames * F
    for j in (n_frames // 4, n_frames // 2 + 1):  # the word of these frames is missing
        a = start + j * F
        x[a:a + Lp] = list(R.psk(M, Lp, rng).astype(np.complex64))
    a = start + (n_frames // 3) * F + F // 2        # a false word inside a payload
    x[a:a + Lp] = list(np.asarray(word))
    del x[start + (2 * n_frames // 3) * F + 3]       # a deleted symbol
    x.insert(start + (5 * n_frames // 6) * F + 5, np.complex64(0.3 - 0.2j))  # an inserted one
    x = np.array(x, np.complex64)
    if special:
        b = start + (n_frames - 3) * F
        x[b + 1] = np.nan
        x[b + Lp + 5] = np.inf
        x[b + F: b + F + Lp] = 0
        x[b + 2 * F + 2: b + 2 * F + 6] = 3e38
    return x


PARAM_SETS = [(0, 1, 0), (1, 1, 2), (3, 3, 1), (0, 3, 4), (2, 2, 0)]  # (V, max_miss, W)


@pytest.mark.parametrize("M", [2, 4, 8])
@pytest.mark.parametrize("V,mm,W", PARAM_SETS)
def test_model_equals_scalar_restatement(M, V, mm, W):
    rng = np.random.default_rng(10 * M + V + 7 * W + mm)
    Lp, F = 13, 13 + 2 * W + 9
    w = R.word(Lp, rng, M)
    x = eventful(w, F, M, 24, rng, W)
    prm = (F, M, 0.6, 0.4, V, mm, W)
    sc = Scalar(w, prm)
    for v in x:
        sc.push(v)
    pay, recs = R.model([x], w, prm)
    want = np.array(sc.recs, R.REC)
    assert len(recs[0]) == len(want) and recs[0].tobytes() == want.tobytes()
    got = pay[0]
    ref = np.array(sc.out, np.complex64)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    ch = R.Channel(w, prm)
    ch.feed(x)
    # a searching channel reports the next position it will search
    pos = max(sc.pos, len(x) - Lp + 1) if sc.state == R.SEARCH else sc.pos
    assert ch.state_tuple() == (sc.state, sc.cnt, pos, sc.R, len(x), sc.payload)


def test_every_record_kind_and_transition():
    """the eventful streams over the parameter sets reach every kind, emitted and not"""
    kinds, emitted = set(), set()
    for M in (2, 4, 8):
        for V, mm, W in PARAM_SETS:
            rng = np.random.default_rng(10 * M + V + 7 * W + mm)
            Lp, F = 13, 13 + 2 * W + 9
            w = R.word(Lp, rng, M)
            _, recs = R.model([eventful(w, F, M, 24, rng, W)], w, (F, M, 0.6, 0.4, V, mm, W))
            kinds |= set(int(k) for k in recs[0]["kind"])
            emitted |= set(int(k) for k, o in zip(recs[0]["kind"], recs[0]["out_index"]) if o != R.NO_OUT)
    assert kinds == {1, 2, 3, 4, 5, 6}
    assert emitted == {R.HIT, R.VERIFY_PASS, R.LOCK_PASS, R.LOCK_MISS}


# ---- bounds and blocking --------------------------------------------------------------------------------------------

def adversarial(kind, word, F, W, n_frames, rng):
    """streams that maximise records or payload: 'pass' plants the word at e - W every frame (LOCK_PASS as early as
    allowed, overlapping payloads when Lp < W); 'restart' plants a word, leaves the next frame without one and plants
    the next word right after the search restarts at e + W + 1"""
    Lp = len(word)
    n = n_frames * F + 4 * F
    x = (R.psk(4, n, rng) * 0.05).astype(np.complex64)
    s = int(rng.integers(0, 8))
    while s + Lp < n:
        x[s:s + Lp] = word
        if kind == "pass":
            s += F - W
        else:
            s += F + W + 1
    return x


def blockings(n, rng):
    yield [n]
    yield [1] * n
    for _ in range(3):
        cuts = np.sort(rng.choice(np.arange(1, n), size=min(n - 1, int(rng.integers(1, 40))), replace=False))
        yield list(np.diff(np.concatenate([[0], cuts, [n]])))


@pytest.mark.parametrize("Lp,W,V,mm", [(8, 32, 0, 3), (8, 32, 1, 1), (16, 4, 1, 2), (13, 0, 0, 1), (32, 1, 3, 2)])
@pytest.mark.parametrize("kind", ["pass", "restart", "noise"])
def test_max_output_never_exceeded(Lp, W, V, mm, kind):
    rng = np.random.default_rng(Lp * 100 + W + V)
    F = Lp + 2 * W + 1
    w = R.word(Lp, rng)
    prm = (F, 4, 0.5, 0.5, V, mm, W)
    x = adversarial(kind, w, F, W, 40, rng) if kind != "noise" else R.psk(4, 40 * F, rng).astype(np.complex64)
    ch = R.Channel(w, prm)
    whole_pay, whole_rec = ch.feed(x)
    bp, br = R.max_output(len(x), 0, Lp, F, W)
    assert len(whole_pay) <= bp and len(whole_rec) <= br
    worst_r = 0.0
    for parts in blockings(len(x), rng):
        ch = R.Channel(w, prm)
        at, pays, recs = 0, [], []
        for m in parts:
            p, r = ch.feed(x[at:at + m])
            bp, br = R.max_output(m, at, Lp, F, W)
            assert len(p) <= bp and len(r) <= br, (m, at, len(p), bp, len(r), br)
            worst_r = max(worst_r, len(r) / max(br, 1))
            pays.append(p)
            recs.append(r)
            at += m
        # the model's outputs do not depend on the blocking
        assert np.concatenate(pays).tobytes() == whole_pay.tobytes()
        assert np.concatenate(recs).tobytes() == whole_rec.tobytes()
    if kind != "noise":
        assert worst_r > 0.45  # the streams come within a factor of about 2 of the record bound


def test_model_split_invariance_multichannel():
    rng = np.random.default_rng(5)
    words = np.stack([R.word(16, rng) for _ in range(3)])
    params = [(60, 4, 0.6, 0.4, 1, 2, 3), (41, 2, 0.6, 0.4, 0, 1, 0), (70, 8, 0.6, 0.4, 3, 3, 1)]
    rows = [eventful(words[k], params[k][0], params[k][1], 20, rng, params[k][6], special=k != 1) for k in range(3)]
    want = R.model(rows, words, params)
    b = R.Bank(words, params)
    got = [[], []]
    at = [0, 0, 0]
    while any(a < len(r) for a, r in zip(at, rows)):
        take = [int(rng.integers(0, 70)) for _ in range(3)]
        p, r = b.feed([row[a:a + t] for row, a, t in zip(rows, at, take)])
        got[0].append(p)
        got[1].append(r)
        at = [a + t for a, t in zip(at, take)]
    for k in range(3):
        assert np.concatenate([p[k] for p in got[0]]).tobytes() == want[0][k].tobytes()
        assert np.concatenate([r[k] for r in got[1]]).tobytes() == want[1][k].tobytes()


# ---- detection statistics (the GPU bars) ----------------------------------------------------------------------------

# Lp = 64 QPSK: rho on random positions is close to exponential with mean 1 / Lp, so P(rho >= th) ~ exp(-64 th).
FALSE_POSITIONS = 10_000_000
TH_SEARCH, TH_CHECK = 0.35, 0.2
ESN0_ACQ = {6.0: 1.0, 3.0: 1.0, 0.0: 0.99}   # Es/N0 dB -> least fraction of frames emitted with LOCK_PASS


def test_false_hits_on_random_qpsk():
    rng = np.random.default_rng(6)
    w = R.word(64, rng)
    Ep = R.energy(w)
    above = {0.1: 0, 0.2: 0, TH_CHECK: 0, TH_SEARCH: 0}
    top = 0.0
    done = 0
    while done < FALSE_POSITIONS:
        n = min(2_000_000, FALSE_POSITIONS - done)
        z = R.psk(4, n + 63, rng).astype(np.complex64)
        _, rho = R.correlate(z, w, Ep)
        for th in above:
            above[th] += int((rho >= th).sum())
        top = max(top, float(rho.max()))
        done += n
    print("false hits over %d positions: %s, largest rho %.4f" % (done, above, top))
    assert above[TH_SEARCH] == 0
    assert 0.2 * done * np.exp(-64 * 0.2) < above[0.2] < 5 * done * np.exp(-64 * 0.2)
    assert 0.5 * done * np.exp(-6.4) < above[0.1] < 2 * done * np.exp(-6.4)


@pytest.mark.parametrize("esn0", sorted(ESN0_ACQ))
def test_detection_and_lock_hold(esn0):
    """Lp = 64 QPSK words, F = 1088, V = 1, max_miss = 3, W = 1: acquisition within V + 2 frames and the fraction of
    later frames emitted with LOCK_PASS (the rest are flywheel frames) over 16 channels of 120 frames"""
    rng = np.random.default_rng(int(esn0 * 10) + 100)
    F, Lp = 1088, 64
    w = R.word(Lp, rng)
    prm = (F, 4, TH_SEARCH, TH_CHECK, 1, 3, 1)
    worst_pass, worst_acq, lost = 1.0, 0, 0
    for k in range(16):
        rot = int(rng.integers(0, 4))
        start = int(rng.integers(0, F))
        x, pays = R.framed(w, F, 120, 4, rng, rot, esn0, start)
        pay, recs = R.model([x], w, prm)
        r = recs[0]
        emitted = r[r["out_index"] != R.NO_OUT]
        first = (int(emitted["pos"][0]) - start) // F
        worst_acq = max(worst_acq, first)
        later = r[(r["kind"] == R.LOCK_PASS) | (r["kind"] == R.LOCK_MISS) | (r["kind"] == R.LOCK_LOST)]
        worst_pass = min(worst_pass, float((later["kind"] == R.LOCK_PASS).mean()))
        lost += int((r["kind"] == R.LOCK_LOST).sum())
        # locked frames sit on the planted words and carry the rotation
        ok = emitted[emitted["kind"] != R.LOCK_MISS]
        assert ((ok["pos"].astype(np.int64) - start) % F == 0).all() and (ok["rot"] == rot).all()
    print("Es/N0 %.0f dB: acquisition by frame %d, worst LOCK_PASS share %.4f, %d losses" % (esn0, worst_acq,
                                                                                          worst_pass, lost))
    assert worst_acq <= 2 and worst_pass >= ESN0_ACQ[esn0] and lost == 0

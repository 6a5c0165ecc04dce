"""CPU: the adaptive equalizer bank's reference model (eq_ref) and ABI without a device.  create rejects every invalid
parameter and fails with NO_DEVICE for a valid one; NULL handles give NULL_HANDLE and the lifecycle contract of the
other handles holds; the vectorised float32 model equals a literal scalar restatement (np.float32 scalars, one tap at
a time) bit for bit; the DD decision's signed-zero and |re| = |im| edges, and non-finite inputs skipping the update;
on the multipath workload the model equalises BPSK, QPSK and 8PSK at the bars the GPU tests use."""
import ctypes as C

import numpy as np
import pytest

import eq_ref as R

F32 = np.float32

# The multipath workload and bars of test_gpu_eq.py: per channel a 0.25 pre-cursor, the main tap and a 0.4
# post-cursor with random phases, normalised, Es/N0 = 30 dB; N = 11 from the centre spike, mu = 5e-3, a = 1,
# err_max = 2; 10 000 symbols, metrics over the last 4000.  Worst over 64 channels per order of this model
# (ISI in dB, EVM): QPSK CMA -36.0 / 0.054, QPSK DD from 4000 -38.1 / 0.066, 8PSK CMA -37.0 / 0.055,
# 8PSK DD from 4000 -38.9 / 0.057, BPSK CMA -6.5 / 0.48, BPSK DD from 4000 -33.1 / 0.089; the input's worst ISI is
# -6.5 dB.  The bars add about 3 dB and 0.02 of margin.  CMA with p = 2 does not equalise BPSK (a non-circular
# constellation): BPSK needs the switch to DD, and its CMA-only bars only say that CMA does not make the input worse.
NTAPS, MU, RADIUS, EMAX, SWITCH = 11, 5e-3, 1.0, 2.0, 4000
NSYM, TAIL, ESN0 = 10000, 4000, 30.0
# (order, S) -> (ISI bar in dB, EVM bar)
BARS = {(4, None): (-33.0, 0.075), (4, SWITCH): (-35.0, 0.085), (8, None): (-34.0, 0.075), (8, SWITCH): (-35.0, 0.08),
        (2, None): (-3.0, 0.7), (2, SWITCH): (-30.0, 0.11)}
INPUT_ISI_WORST = -6.5


def adapt_for(M, S):
    return (M, MU, RADIUS, EMAX, S)


def workload_metrics(y, taps, h, a):
    """per channel (ISI in dB, EVM) over the last TAIL symbols"""
    isi = np.array([R.isi_db(taps[k], h[k]) for k in range(len(h))])
    ev = np.array([R.evm(y[k], taps[k], h[k], a[k], NSYM - TAIL) for k in range(len(h))])
    return isi, ev


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---- a literal restatement: one channel, np.float32 scalars, one tap at a time ------------------------------------

def scalar_model(x, N, adapt, taps0):
    M, mu, a, emax, S = adapt
    mu, a, emax = F32(mu), F32(a), F32(emax)
    S = R.CMA_ONLY if S is None else S
    R2 = a * a
    dp, dq = R.decision_points(M, a)
    W = R.lanes(N)
    wr = [F32(v.real) for v in taps0]
    wi = [F32(v.imag) for v in taps0]
    line = [(F32(0), F32(0))] * N
    ys, es = [], []
    with np.errstate(all="ignore"):
        for s, xs in enumerate(x):
            line = [(F32(xs.real), F32(xs.imag))] + line[:-1]
            P = []
            for j in range(N):
                xr, xi = line[j]
                P.append((wr[j] * xr - wi[j] * xi, wr[j] * xi + wi[j] * xr))
            p = []
            for l in range(W):
                if l >= N:
                    p.append((F32(0), F32(0)))
                elif l + 32 < N:
                    p.append((P[l][0] + P[l + 32][0], P[l][1] + P[l + 32][1]))
                else:
                    p.append(P[l])
            o = W // 2
            while o >= 1:
                for l in range(o):
                    p[l] = (p[l][0] + p[l + o][0], p[l][1] + p[l + o][1])
                o //= 2
            yr, yi = p[0]
            if s < S:
                eps = (yr * yr + yi * yi) - R2
                gr, gi = eps * yr, eps * yi
            else:
                if M == 2 or abs(yr) >= abs(yi):
                    da, db = dp, dq
                else:
                    da, db = dq, dp
                gr = yr - (da if yr >= 0 else -da)
                gi = yi - (db if yi >= 0 else -db)
            ys.append((yr, yi))
            if not (np.isfinite(yr) and np.isfinite(yi) and np.isfinite(gr) and np.isfinite(gi)):
                es.append((F32(0), F32(0)))
                continue
            er = min(max(gr, -emax), emax)
            ei = min(max(gi, -emax), emax)
            es.append((F32(er), F32(ei)))
            ur, ui = mu * er, mu * ei
            for j in range(N):
                xr, xi = line[j]
                wr[j] = wr[j] - (ur * xr + ui * xi)
                wi[j] = wi[j] - (ui * xr - ur * xi)
    y = R.complex_parts(np.array([v[0] for v in ys], F32), np.array([v[1] for v in ys], F32))
    e = R.complex_parts(np.array([v[0] for v in es], F32), np.array([v[1] for v in es], F32))
    return y, e, R.complex_parts(np.array(wr, F32), np.array(wi, F32))


@pytest.mark.parametrize("N", [1, 2, 5, 16, 32, 33, 64])
def test_model_equals_scalar_restatement(N):
    """three channels: CMA only, DD only and a switch mid-stream, orders 4, 8 and 2; random taps and inputs"""
    rng = np.random.default_rng(N)
    L = 120
    x = ((rng.standard_normal((3, L)) + 1j * rng.standard_normal((3, L))) * 0.7).astype(np.complex64)
    t0 = ((rng.standard_normal((3, N)) + 1j * rng.standard_normal((3, N))) / N).astype(np.complex64)
    t0[0, (N - 1) // 2] += 1
    adapts = [(4, 0.01, 1.0, 2.0, None), (8, 0.02, 1.5, 1.0, 0), (2, 0.015, 0.8, 0.5, 57)]
    y, e, taps = R.model(x, N, adapts, t0)
    for k in range(3):
        ys, es, ts = scalar_model(x[k], N, adapts[k], t0[k])
        assert np.array_equal(_bits(y[k]), _bits(ys)), k
        assert np.array_equal(_bits(e[k]), _bits(es)), k
        assert np.array_equal(_bits(taps[k]), _bits(ts)), k
    assert (np.abs(taps - t0) > 0).any()


def test_centre_spike_at_mu_zero_delays():
    for N in (1, 2, 7, 11, 32, 64):
        x = (np.arange(1, 301) * (1 + 0.5j)).astype(np.complex64)[None]
        y, _, taps = R.model(x, N, (4, 0.0, 1.0, 2.0, None))
        c = (N - 1) // 2
        assert np.array_equal(_bits(y[0, c:]), _bits(x[0, :300 - c])) and (y[0, :c] == 0).all()
        assert np.array_equal(taps[0], R.centre_spike(N))


def test_decision_edges():
    """sgn(-0) = +1; |re| = |im| takes the first form for M = 8; M = 2 always takes (+-a, 0)"""
    A = R.Adapt([(2, 0.0, 2.0, 10.0, 0), (4, 0.0, 2.0, 10.0, 0), (8, 0.0, 2.0, 10.0, 0)], 3)
    p, q = R.decision_points(8, 2.0)
    c = F32(2.0 / np.sqrt(2.0))
    assert p == F32(2.0 * np.cos(np.pi / 8)) and q == F32(2.0 * np.sin(np.pi / 8))
    s = np.zeros(3, np.uint64)
    cases = [(F32(-0.0), F32(-0.0)), (F32(0.5), F32(-0.5)), (F32(-0.25), F32(3.0)), (F32(-0.0), F32(-1.0))]
    for yr0, yi0 in cases:
        yr, yi = np.full(3, yr0), np.full(3, yi0)
        er, ei, ok = R.error(yr, yi, s, A)
        assert ok.all()
        sr, si = (1 if yr0 >= 0 else -1), (1 if yi0 >= 0 else -1)
        assert er[0] == yr0 - sr * F32(2.0) and _bits(ei[0:1]) == _bits(np.array([yi0 - F32(0.0)], F32))
        assert er[1] == yr0 - sr * c and ei[1] == yi0 - si * c
        first = abs(yr0) >= abs(yi0)
        assert er[2] == yr0 - sr * (p if first else q) and ei[2] == yi0 - si * (q if first else p)
    # -0 is +1: y = (-0, -0) decides (+a, 0) for BPSK, so e = (-a, -0)
    er, ei, _ = R.error(np.full(3, F32(-0.0)), np.full(3, F32(-0.0)), s, A)
    assert er[0] == -2.0 and np.signbit(ei[0])


def test_non_finite_skips_the_update():
    """a NaN or Inf symbol: the N outputs whose delay line holds it are not finite, their e is 0 and the taps do not
    change across them; the outputs before are those of the clean run bit for bit"""
    N, L, m = 7, 400, 150
    rng = np.random.default_rng(3)
    x = ((rng.standard_normal((2, L)) + 1j * rng.standard_normal((2, L))) * 0.7).astype(np.complex64)
    bad = x.copy()
    bad[0, m] = complex(np.nan, 0.0)
    bad[1, m] = complex(1.0, np.inf)
    ad = (4, 0.01, 1.0, 2.0, 100)
    y, e, _ = R.model(bad, N, ad)
    yc, ec, _ = R.model(x, N, ad)
    for k in range(2):
        assert np.array_equal(_bits(y[k, :m]), _bits(yc[k, :m])) and np.array_equal(_bits(e[k, :m]), _bits(ec[k, :m]))
        assert all(not np.isfinite(v) for v in y[k, m:m + N]) and (e[k, m:m + N] == 0).all()
        assert np.isfinite(y[k, m + N:]).all() and np.isfinite(e[k]).all()
    # the taps after the N skipped symbols equal those before them
    _, _, t_before = R.model(bad[:, :m], N, ad)
    _, _, t_after = R.model(bad[:, :m + N], N, ad)
    assert np.array_equal(_bits(t_before), _bits(t_after))


def test_model_equalises_the_workload():
    """64 channels per order and adaptation, on the multipath workload: within the bars (worst over channels)"""
    rng = np.random.default_rng(17)
    cases = list(BARS)
    xs, hs, as_ = [], [], []
    for M, S in cases:
        x, h, a = R.multipath_rows(M, 64, NSYM, ESN0, rng)
        xs.append(x)
        hs.append(h)
        as_.append(a)
    x = np.concatenate(xs)
    adapts = [adapt_for(M, S) for M, S in cases for _ in range(64)]
    y, _, taps = R.model(x, NTAPS, adapts)
    for i, (M, S) in enumerate(cases):
        sl = slice(64 * i, 64 * (i + 1))
        isi, ev = workload_metrics(y[sl], taps[sl], hs[i], as_[i])
        assert max(R.isi_db(R.centre_spike(NTAPS), h) for h in hs[i]) <= INPUT_ISI_WORST + 0.5
        bar_isi, bar_evm = BARS[(M, S)]
        print("M = %d, S = %s: ISI worst %.1f median %.1f dB, EVM worst %.3f median %.3f"
              % (M, S, isi.max(), np.median(isi), ev.max(), np.median(ev)))
        assert isi.max() < bar_isi and ev.max() < bar_evm, (M, S, isi.max(), ev.max())


# ---- the ABI without a device ------------------------------------------------------------------------------------

def _cfg(sdr, N, adapts, C_, taps=None, n_tap_sets=None, n_adapt=None):
    """the config keeps its arrays alive"""
    F = sdr._ffi
    ad = None if adapts is None else (F.EqAdapt * len(adapts))(
        *[F.EqAdapt(a[0], a[1], a[2], a[3], R.CMA_ONLY if a[4] is None else a[4]) for a in adapts])
    t = None if taps is None else np.ascontiguousarray(np.asarray(taps, np.complex64))
    cfg = F.EqConfig(N, None if t is None else t.ctypes.data,
                     (0 if t is None else t.size // max(N, 1)) if n_tap_sets is None else n_tap_sets,
                     None if ad is None else C.addressof(ad), (0 if adapts is None else len(adapts))
                     if n_adapt is None else n_adapt, C_, 0, None)
    cfg.keep = (ad, t)
    return cfg


def test_eq_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    ok = (4, 5e-3, 1.0, 2.0, 4000)
    nan, inf = float("nan"), float("inf")
    bad_adapts = [(3, 5e-3, 1.0, 2.0, 0), (0, 5e-3, 1.0, 2.0, 0), (16, 5e-3, 1.0, 2.0, 0),
                  (4, -1e-3, 1.0, 2.0, 0), (4, nan, 1.0, 2.0, 0), (4, inf, 1.0, 2.0, 0),
                  (4, 5e-3, 0.0, 2.0, 0), (4, 5e-3, -1.0, 2.0, 0), (4, 5e-3, nan, 2.0, 0), (4, 5e-3, inf, 2.0, 0),
                  (4, 5e-3, 2e19, 2.0, 0),      # fl(a a) overflows
                  (4, 5e-3, 1.0, 0.0, 0), (4, 5e-3, 1.0, -2.0, 0), (4, 5e-3, 1.0, nan, 0), (4, 5e-3, 1.0, inf, 0)]
    assert lib.sdr_eq_create(None, C.byref(err)) is None and err.value == 100
    good4 = np.ones((4, 5), np.complex64)
    bad_taps = good4.copy()
    bad_taps[2, 3] = complex(0.0, np.nan)
    inf_taps = good4.copy()
    inf_taps[0, 0] = complex(np.inf, 0.0)
    bad = [_cfg(sdr, 5, None, 4, n_adapt=1),                       # NULL adapt
           _cfg(sdr, 0, [ok], 4),                                   # N = 0
           _cfg(sdr, 65, [ok], 4),                                  # N > 64
           _cfg(sdr, 5, [ok], 0),                                   # C = 0
           _cfg(sdr, 5, [ok], 65537),                               # C > 65536
           _cfg(sdr, 5, [ok, ok], 4),                               # n_adapt not 1 or C
           _cfg(sdr, 5, [ok], 4, taps=np.ones((2, 5)), n_tap_sets=2),  # n_tap_sets not 0, 1 or C
           _cfg(sdr, 5, [ok], 4, n_tap_sets=1),                     # NULL taps
           _cfg(sdr, 5, [ok], 4, n_tap_sets=4),                     # NULL taps
           _cfg(sdr, 5, [ok], 4, taps=bad_taps),                    # NaN tap
           _cfg(sdr, 5, [ok], 4, taps=inf_taps)]                    # Inf tap
    bad += [_cfg(sdr, 5, [ok] * 3 + [a], 4) for a in bad_adapts]
    bad += [_cfg(sdr, 5, [a], 1) for a in bad_adapts]
    for i, cfg in enumerate(bad):
        err.value = 0
        assert lib.sdr_eq_create(C.byref(cfg), C.byref(err)) is None and err.value == 100, i
    n = np.zeros(4, np.uintp)
    w = np.zeros(64, np.complex64)
    assert lib.sdr_eq_process(None, None, n.ctypes.data, 0, None, None, 0) == 103
    assert lib.sdr_eq_process_dev(None, None, n.ctypes.data, 0, None, None, 0) == 103
    assert lib.sdr_eq_get_taps(None, 0, w.ctypes.data) == 103
    assert lib.sdr_eq_reset(None) == 103
    assert lib.sdr_eq_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_eq_destroy(None)
    if sdr.device_count() == 0:
        # valid, at the edges: N = 1 and 64, C = 65536, every order, mu = 0, shared and per-channel taps and adaptation
        edge = [(2, 0.0, 1e-3, 1e-30, 0), (4, 1.0, 1e18, 1e30, None), (8, 5e-3, 1.0, 2.0, 1), (4, 5e-3, 1.0, 2.0, 7)]
        for cfg in [_cfg(sdr, 1, [ok], 1), _cfg(sdr, 64, edge, 4, taps=np.ones((4, 64))),
                    _cfg(sdr, 11, [ok], 65536, taps=np.ones(11)), _cfg(sdr, 33, edge, 4)]:
            err.value = 0
            assert lib.sdr_eq_create(C.byref(cfg), C.byref(err)) is None and err.value == 102
            assert lib.sdr_eq_create(C.byref(cfg), None) is None


def test_eq_lifecycle_contract(sdr):
    """the contract test_handle_lifecycle_host.py checks for every other handle: a NULL configuration is INVALID_ARG
    and a NULL err is accepted; a valid one is NO_DEVICE without a GPU; clone and reset of NULL give NULL_HANDLE;
    destroy of NULL is a no-op"""
    lib = sdr.lib()
    err = C.c_int(-1)
    assert lib.sdr_eq_create(None, C.byref(err)) is None and err.value == 100
    assert lib.sdr_eq_create(None, None) is None
    if sdr.device_count() == 0:
        cfg = _cfg(sdr, 11, [(4, 5e-3, 1.0, 2.0, None)], 2)
        err.value = -1
        assert lib.sdr_eq_create(C.byref(cfg), C.byref(err)) is None and err.value == 102
        assert lib.sdr_eq_create(C.byref(cfg), None) is None
    err.value = -1
    assert lib.sdr_eq_clone(None, C.byref(err)) is None and err.value == 103
    assert lib.sdr_eq_clone(None, None) is None
    assert lib.sdr_eq_reset(None) == 103
    lib.sdr_eq_destroy(None)


def test_eq_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Eq(11, (4, 5e-3, 1.0, 2.0, None), n_channels=3)
    assert e.value.code == 102

"""Symbol timing recovery bank (sdr_tsync): the loop's integer recurrence replayed exactly from the reported errors;
every symbol against the f64 interpolant at its exact position and every error against the float32 detector on the f64
mid sample; spot symbols, mid samples and errors equal to sdr_arb's outputs bit for bit; the open loop is sdr_arb;
acquisition and tracking of RRC-shaped QPSK at known clock offsets and delays, and saturation of v at +-V; blockings,
clones, resets, retries, strides and host against device give the same bits; NaN bounds; the launch count; the
device-resident sdr_ddc -> sdr_tsync chain; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import arb_ref as A
import gen
import tsync_ref as R
from test_tsync_host import ACQ, BAR_EVM, BAR_PPM, BAR_TIMING

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ONE = A.ONE
F32 = np.float32

PERIODS = [2 * ONE, A.step_of(2 * (1 + 37e-6), 1.0), A.step_of(4.41, 1.0), 8 * ONE, A.step_of(10.3, 1.0)]
LOOPS = [(0.05, 0.002, 1.0, 0.01), (0.2, 0.01, 2.0, 0.05), (0.0, 0.0, 1.0, 0.0), (0.02, 0.0005, 0.5, 0.25)]
BETA, SPAN = 0.35, 8


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _taps(C_, L, P, shared, seed=0):
    """low-pass prototypes at P times the input rate with sum P, one row per channel unless shared"""
    rng = np.random.default_rng(seed)
    rows = []
    for _ in range(1 if shared else C_):
        t = gen.lowpass_taps(L, (0.3 + 0.1 * rng.random()) / P, 1.0).astype(np.float64) if L > 2 else np.ones(L)
        rows.append(P * t / t.sum())
    t = np.asarray(rows, np.float32)
    return t[0] if shared else t


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n)


def _firsts(C_, seed):
    rng = np.random.default_rng(seed)
    return [[0, int(rng.integers(0, 1 << 62)) % (3 * ONE), (int(rng.integers(0, 40)) << 64) | 12345][k % 3]
            for k in range(C_)]


def _z64(h, P, row, taus):
    """the f64 interpolant (computed form, exact weights) at exact positions"""
    if not taus:
        return np.zeros(0, np.complex128)
    at = max(0, (min(taus) >> 64) - -(-h.size // P) - 1)
    end = (max(taus) >> 64) + 1
    return A.computed_f64(h, P, np.asarray(row[at:end], np.complex128), taus, at=at)


def _detector(y, yp, m, emax):
    """the float32 detector, vectorised: every operation rounded in f32, clamped, 0 where not finite"""
    y, yp, m = (np.asarray(x, np.complex64) for x in (y, yp, m))
    with np.errstate(all="ignore"):
        g = (y.real - yp.real) * m.real + (y.imag - yp.imag) * m.imag
        e = np.minimum(np.maximum(g, -F32(emax)), F32(emax)).astype(np.float32)
    return np.where(np.isfinite(g), e, F32(0)).astype(np.float32)


def _loop_of(loops, k):
    lp = loops if np.ndim(loops[0]) == 0 else loops[k]
    return tuple(F32(x) for x in lp[:3]) + (float(lp[3]),)


def _check_exact(sdr, ts, h, P, y, periods, firsts, loops, sym, pos, err, spot_channels):
    """replay, f64 bars and the sdr_arb spot identity for every channel of one process() over rows y"""
    C_ = len(sym)
    nf = y.shape[1]
    for k in range(C_):
        T, lp, hk = periods[k], _loop_of(loops, k), A.taps_of(h, k).astype(np.float64)
        n = len(pos[k])
        assert n > 0 and (pos[k][-1] >> 64) < nf
        vs, nxt = R.replay(pos[k], err[k], T, lp, first=firsts[k])
        assert (nxt[0] >> 64) >= nf and ts.state(k) == nxt, k
        z64 = _z64(hk, P, y[k], pos[k])
        M = max(np.abs(z64).max(), 1e-30)
        assert np.abs(sym[k] - z64).max() <= 1e-5 * M, k
        mids = [R.mid_of(pos[k][s], vs[s], T) for s in range(1, n)]
        assert all(m >= p for m, p in zip(mids, pos[k]))
        m64 = _z64(hk, P, y[k], mids)
        want = _detector(sym[k][1:], sym[k][:-1], m64, lp[2])
        M2 = max(M, np.abs(m64).max() if mids else 0) ** 2
        assert err[k][0] == 0 and np.abs(err[k][1:] - want).max(initial=0) <= 1e-4 * M2, k
    # spot symbols and mid samples: sdr_arb's outputs at those positions, and the errors from them, bit for bit
    for k in spot_channels:
        T, lp = periods[k], _loop_of(loops, k)
        vs, _ = R.replay(pos[k], err[k], T, lp, first=firsts[k])
        n = len(pos[k])
        ss = sorted(set(np.linspace(1, n - 1, min(64, n - 1)).astype(int).tolist()))
        taus = [pos[k][s] for s in ss] + [R.mid_of(pos[k][s], vs[s], T) for s in ss]
        arb = sdr.Arb(A.taps_of(h, k), P, ONE, taus)
        z = arb.process(np.repeat(y[k][None], len(taus), axis=0))
        ya = np.array([z[j][0] for j in range(len(ss))], np.complex64)
        ma = np.array([z[len(ss) + j][0] for j in range(len(ss))], np.complex64)
        assert np.array_equal(_bits(ya), _bits(sym[k][ss])), k
        e = _detector(sym[k][ss], sym[k][[s - 1 for s in ss]], ma, lp[2])
        assert np.array_equal(_bits(e), _bits(err[k][ss])), k


@pytest.mark.parametrize("C_,P,L,shared_taps,shared_loops", [
    (1, 32, 8193, True, True), (1, 256, 4097, True, True), (1, 1, 1, True, True), (3, 1, 7, False, False),
    (3, 256, 2049, False, True), (17, 32, 255, True, False), (17, 1, 33, False, False), (256, 32, 513, True, False),
    (256, 256, 8193, False, True), (1024, 32, 255, True, False), (1024, 1, 15, False, True)])
def test_tsync_exact_loop_arithmetic(sdr, C_, P, L, shared_taps, shared_loops):
    periods = [PERIODS[(k + L) % len(PERIODS)] for k in range(C_)]
    firsts = _firsts(C_, C_ + L)
    loops = LOOPS[L % len(LOOPS)] if shared_loops else [LOOPS[k % len(LOOPS)] for k in range(C_)]
    h = _taps(C_, L, P, shared_taps, C_ + P)
    nf = 4000 if C_ <= 17 else 400
    y = _rows(C_, nf, C_ + L + P) * 2
    ts = sdr.Tsync(h, P, periods, loops, firsts)
    cap = ts.max_output(nf)
    for k in range(C_):
        assert cap[k] == R.max_output(nf, periods[k], _loop_of(loops, k))
    sym, pos, err = ts.process(y)
    for k in range(C_):
        assert len(sym[k]) <= cap[k]
    spot = sorted({0, C_ - 1})
    _check_exact(sdr, ts, h, P, y, periods, firsts, loops, sym, pos, err, spot)


def test_tsync_open_loop_is_arb(sdr):
    """kp = ki = 0: sdr_arb's outputs and counts at step T and first tau(0), bit for bit"""
    C_, P, L = 5, 32, 1023
    periods = PERIODS
    firsts = _firsts(C_, 3)
    h = _taps(C_, L, P, False, 4)
    y = _rows(C_, 5000, 5)
    sym, pos, err = sdr.Tsync(h, P, periods, (0.0, 0.0, 1.0, 0.0), firsts).process(y)
    for k in range(C_):
        z = sdr.Arb(h[k], P, periods[k], firsts[k]).process(y[k])[0]
        assert len(sym[k]) == z.size == A.released(5000, firsts[k], periods[k])
        assert np.array_equal(_bits(sym[k]), _bits(z))
        assert pos[k] == [firsts[k] + r * periods[k] for r in range(z.size)]


def _qpsk_bank(periods_f, ppms, n_sym, P, seed):
    """RRC QPSK rows at the given nominal periods and clock offsets, random delays, Es/N0 = 30 dB; the matched filters
    zero-padded to one length.  Returns rows, true periods, delays, taps [C, L], filter centres."""
    rng = np.random.default_rng(seed)
    rows, trues, delays, taps, centres = [], [], [], [], []
    for per, ppm in zip(periods_f, ppms):
        true = per * (1 + ppm)
        d = rng.uniform(0, true)
        y, _ = R.qpsk_channel(int(n_sym * true), true, d, BETA, SPAN, 30.0, rng)
        h, c = R.rrc_taps(per, P, BETA, SPAN)
        rows.append(y)
        trues.append(true)
        delays.append(d)
        taps.append(h)
        centres.append(c)
    L = max(t.size for t in taps)
    tp = np.zeros((len(taps), L), np.float32)
    for k, t in enumerate(taps):
        tp[k, :t.size] = t
    return rows, trues, delays, tp, centres


def test_tsync_acquires_and_tracks_qpsk(sdr):
    """256 channels, 2-8 frames per symbol, offsets 0, +-50, +-500 ppm, random delays, Es/N0 = 30 dB, gains from
    sdr_tsync_loop_design (B_n T = 0.01, zeta = 0.707): after ACQ symbols every position lies within BAR_TIMING T of a
    true symbol centre, the EVM after a complex gain fit is below BAR_EVM and mean(T + v) is within BAR_PPM of the true
    period (bars from the CPU model, test_tsync_host.py)"""
    C_, P = 256, 32
    pers = [[2, 2.5, 3, 4, 5, 6, 8][k % 7] for k in range(C_)]
    ppms = [[0, 50e-6, -50e-6, 500e-6, -500e-6][k % 5] for k in range(C_)]
    rows, trues, delays, h, centres = _qpsk_bank(pers, ppms, 3000, P, 31)
    K = R.gardner_slope(BETA)
    loops = [sdr.tsync_loop_design(0.01, 0.707, K, p) + (2.0, 0.01) for p in pers]
    periods = [A.step_of(p, 1.0) for p in pers]
    ts = sdr.Tsync(h, P, periods, loops)
    sym, pos, err = ts.process(rows)
    worst = np.zeros(3)
    for k in range(C_):
        vs, nxt = R.replay(pos[k], err[k], periods[k], _loop_of(loops, k), first=0)
        assert ts.state(k) == nxt
        r = R.tracking(pos[k], sym[k], vs, periods[k], trues[k], delays[k], centres[k], ACQ)
        worst = np.maximum(worst, np.abs(r))
        assert r[0] < BAR_TIMING and r[1] < BAR_EVM and abs(r[2]) < BAR_PPM, (k, pers[k], ppms[k], r)
    print("worst timing %.4f T, EVM %.4f, period %.2f ppm" % (worst[0], worst[1], worst[2] * 1e6))


def test_tsync_offset_beyond_max_dev_saturates(sdr):
    """+-500 ppm against max_dev = 100 ppm: v never passes V and keeps returning to exactly +-V, the sign of the
    offset, after acquisition"""
    P = 32
    pers, ppms = [4, 4, 2.5, 8], [500e-6, -500e-6, 500e-6, -500e-6]
    rows, trues, delays, h, centres = _qpsk_bank(pers, ppms, 3000, P, 32)
    K = R.gardner_slope(BETA)
    loops = [sdr.tsync_loop_design(0.01, 0.707, K, p) + (2.0, 100e-6) for p in pers]
    periods = [A.step_of(p, 1.0) for p in pers]
    ts = sdr.Tsync(h, P, periods, loops)
    sym, pos, err = ts.process(rows)
    for k in range(4):
        V = R.dev_bound(100e-6, periods[k])
        vs, nxt = R.replay(pos[k], err[k], periods[k], _loop_of(loops, k), first=0)
        sign = 1 if ppms[k] > 0 else -1
        assert ts.state(k) == nxt and max(abs(v) for v in vs) == V, k
        assert vs[-ACQ:].count(sign * V) > ACQ // 10, (k, vs[-ACQ:].count(sign * V))


def test_tsync_blockings_clone_reset_retry_strides(sdr):
    C_, P, L = 5, 32, 255
    periods = PERIODS
    firsts = _firsts(C_, 7)
    loops = [LOOPS[k % 2] for k in range(C_)]
    h = _taps(C_, L, P, False, 9)
    nf = 1500
    y = _rows(C_, nf, 10) * 2

    def make(**kw):
        return sdr.Tsync(h, P, periods, loops, firsts, **kw)

    def same(a, b):
        assert np.array_equal(_bits(a[0]), _bits(b[0])) and a[1] == b[1] and np.array_equal(_bits(a[2]), _bits(b[2]))

    def cat(parts, k, lo=0):
        return (np.concatenate([p[0][k] for p in parts]), sum((p[1][k] for p in parts), []),
                np.concatenate([p[2][k] for p in parts]))

    one = make().process(y)
    ref = [(one[0][k], one[1][k], one[2][k]) for k in range(C_)]
    # 1-frame calls
    p = make()
    parts = [p.process(y[:, m:m + 1]) for m in range(300)] + [p.process(y[:, 300:])]
    for k in range(C_):
        same(cat(parts, k), ref[k])
    # random splits, different per channel, with a clone mid-stream
    rng = np.random.default_rng(L)
    p = make()
    at = np.zeros(C_, np.int64)
    parts, clone = [], None
    while (at < nf).any():
        take = np.minimum(nf - at, rng.integers(0, 90, C_))
        parts.append(p.process([y[k, at[k]:at[k] + take[k]] for k in range(C_)]))
        at += take
        if clone is None and at.min() > nf // 2:
            clone, cat_at, made = p.clone(), at.copy(), [sum(len(q[0][k]) for q in parts) for k in range(C_)]
    for k in range(C_):
        same(cat(parts, k), ref[k])
    cz = clone.process([y[k, cat_at[k]:] for k in range(C_)])
    for k in range(C_):
        same((cz[0][k], cz[1][k], cz[2][k]), tuple(r[made[k]:] for r in ref[k]))
    p.reset()
    assert p.state(2) == (firsts[2], 0)
    again = p.process(y)
    for k in range(C_):
        same((again[0][k], again[1][k], again[2][k]), ref[k])
    # a too-small out_cap is refused before any state changes, host and device; the retry gives the same bits
    torch, dev = _torch()
    p = make()
    first = p.process(y[:, :7])
    restm = np.ascontiguousarray(y[:, 7:])
    n = np.full(C_, restm.shape[1], np.uintp)
    cap = int(p.max_output(restm.shape[1]).max())
    sym = np.empty((C_, cap), np.complex64)
    got = np.zeros(C_, np.uintp)
    before = p.state(3)
    rc = sdr.lib().sdr_tsync_process(p.h, restm.ctypes.data, n.ctypes.data, restm.shape[1], sym.ctypes.data, None,
                                     None, cap - 1, cap, got.ctypes.data)
    assert rc == 104 and not got.any()
    d_in = torch.from_numpy(restm).to(dev)
    d_sym = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_tsync_process_dev(p.h, d_in.data_ptr(), n.ctypes.data, restm.shape[1], d_sym.data_ptr(), None,
                                         None, cap - 1, cap, got.ctypes.data)
    assert rc == 104 and not got.any() and p.state(3) == before
    second = p.process(restm)
    for k in range(C_):
        same(cat([first, second], k), ref[k])
    # odd device strides give the host bits, and nothing past the counts is written
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = y
    d_y = torch.from_numpy(pad).to(dev)
    q = make(stream=st)
    cap = int(q.max_output(nf).max())
    d_sym = torch.full((C_, cap + 3), float("nan"), dtype=torch.complex64, device=dev)
    d_pos = torch.zeros((C_, cap + 3, 2), dtype=torch.int64, device=dev)
    d_err = torch.full((C_, cap + 3), float("nan"), dtype=torch.float32, device=dev)
    got = q.process_dev(d_y, nf, nf + 5, d_sym, cap, cap + 3, d_pos, d_err)
    out, po, er = d_sym.cpu().numpy(), d_pos.cpu().numpy().view(np.uint64), d_err.cpu().numpy()
    for k in range(C_):
        g = int(got[k])
        assert g == len(ref[k][0])
        same((out[k, :g], [(int(a) << 64) | int(b) for a, b in po[k, :g]], er[k, :g]), ref[k])
        assert np.isnan(out[k, g:]).all() and np.isnan(er[k, g:]).all()
    # misaligned device pointers are refused
    n = np.full(C_, nf, np.uintp)
    got = np.zeros(C_, np.uintp)
    fresh = make()
    rc = sdr.lib().sdr_tsync_process_dev(fresh.h, d_y.data_ptr() + 4, n.ctypes.data, nf + 5, d_sym.data_ptr(), None,
                                         None, cap + 3, cap + 3, got.ctypes.data)
    assert rc == 105 and not got.any()


def test_tsync_host_call_larger_than_the_chunk(sdr):
    """one host call of more frames than the host path moves per round gives process_dev's bits"""
    torch, dev = _torch()
    C_, P, L = 2, 64, 1024
    periods = [PERIODS[1], PERIODS[2]]
    loops = (0.05, 0.002, 1.0, 0.01)
    h = _taps(1, L, P, True, 12)
    nf = (1 << 21) + 777  # the host path moves 2^21 frames per channel per round at C = 2
    y = _rows(C_, nf, 13) * 2
    host = sdr.Tsync(h, P, periods, loops).process(y)
    st = torch.cuda.current_stream(dev)
    b = sdr.Tsync(h, P, periods, loops, stream=st)
    cap = int(b.max_output(nf).max())
    d_y = torch.from_numpy(y).to(dev)
    d_sym = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_pos = torch.empty((C_, cap, 2), dtype=torch.int64, device=dev)
    d_err = torch.empty((C_, cap), dtype=torch.float32, device=dev)
    got = b.process_dev(d_y, nf, nf, d_sym, cap, cap, d_pos, d_err)
    z, po, er = d_sym.cpu().numpy(), d_pos.cpu().numpy().view(np.uint64), d_err.cpu().numpy()
    for k in range(C_):
        g = int(got[k])
        assert len(host[0][k]) == g
        assert np.array_equal(_bits(host[0][k]), _bits(z[k, :g])) and np.array_equal(_bits(host[2][k]),
                                                                                       _bits(er[k, :g]))
        assert host[1][k] == [(int(a) << 64) | int(c) for a, c in po[k, :g]]
    del d_y, d_sym, d_pos, d_err


@pytest.mark.parametrize("P,L", [(1, 64), (32, 255)])
def test_tsync_nan_poisons_exactly_its_symbols(sdr, P, L):
    C_ = 2
    periods = [PERIODS[2], PERIODS[4]]
    loops = (0.05, 0.002, 1.0, 0.01)
    h = _taps(C_, L, P, False, 20)
    T = -(-L // P)
    nf = 8 * T + 400
    y = _rows(C_, nf, 21) * 2
    m = nf // 2
    bad = y.copy()
    bad[1, m] = np.complex64(complex(np.nan, 0.0))
    sym, pos, err = sdr.Tsync(h, P, periods, loops).process(bad)
    ref = sdr.Tsync(h, P, periods, loops).process(y)
    assert np.array_equal(_bits(sym[0]), _bits(ref[0][0])) and pos[0] == ref[1][0]
    hit = np.array([(t >> 64) - A.terms(P, L, t) + 1 <= m <= (t >> 64) for t in pos[1]])
    assert hit.any() and not hit.all()
    assert np.isnan(sym[1][hit].real).all() and np.isfinite(sym[1][~hit]).all()
    assert np.isfinite(err[1]).all()
    idx = np.nonzero(hit)[0]
    assert (err[1][idx] == 0).all() and (err[1][idx[-1] + 1] == 0) and idx[-1] + 2 < len(sym[1])
    R.replay(pos[1], err[1], periods[1], _loop_of(loops, 1), first=0)
    # before the NaN's first symbol the channel is unchanged
    s0 = idx[0]
    assert np.array_equal(_bits(sym[1][:s0]), _bits(ref[0][1][:s0])) and pos[1][:s0 + 1] == ref[1][1][:s0 + 1]


@pytest.mark.parametrize("C_", [1, 1024])
def test_tsync_launch_count(sdr, C_):
    torch, dev = _torch()
    periods = [PERIODS[k % len(PERIODS)] for k in range(C_)]
    b = sdr.Tsync(_taps(1, 255, 32, True, 22), 32, periods, LOOPS[0])
    n = 2000
    d_y = torch.randn((C_, n), dtype=torch.complex64, device=dev)
    cap = int(b.max_output(n).max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    before = sdr.kernel_launch_count()
    got = b.process_dev(d_y, n, n, d_z, cap, cap)
    assert sdr.kernel_launch_count() - before <= 2 and got.min() > 0


def test_ddc_to_tsync_chain(sdr):
    """four RRC QPSK channels (64 input samples per symbol, offsets 0, +50, -500, +500 ppm) at different frequencies in
    one u8 IQ capture -> sdr_ddc (u8, tensor path, D = 16) -> sdr_tsync at 4 frames per symbol, device-resident: equal
    to the host-hop chain bit for bit, and tracking within the bars (the DDC puts input time t at output frame
    (t - (D - 1) + (Ld - 1) / 2) / D)"""
    torch, dev = _torch()
    n, D, Ld = 1 << 22, 16, 255
    freqs = [0.1, -0.27, 0.3, -0.05]
    ppms = [0.0, 50e-6, -500e-6, 500e-6]
    rng = np.random.default_rng(40)
    x = np.zeros(n, np.complex128)
    delays = []
    for f, ppm in zip(freqs, ppms):
        d = rng.uniform(0, 64)
        s, _ = R.qpsk_channel(n, 64 * (1 + ppm), d, BETA, SPAN, 80.0, rng)
        x += s * np.exp(2j * np.pi * f * np.arange(n))
        delays.append(d)
    raw = np.empty(2 * n, np.uint8)
    raw[0::2] = np.clip(np.round(128 + 12 * x.real), 0, 255)
    raw[1::2] = np.clip(np.round(128 + 12 * x.imag), 0, 255)
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0)
    st = torch.cuda.current_stream(dev)
    ddc = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    nf = n // D
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((4, nf), dtype=torch.complex64, device=dev)
    assert ddc.process_dev(d_in, n, d_y, nf, nf) == nf
    assert ddc.last_path == 2
    yh = d_y.cpu().numpy()
    P = 32
    h, c = R.rrc_taps(4.0, P, BETA, SPAN)
    taps = np.stack([h / np.sqrt((np.abs(yh[k]) ** 2).mean()) for k in range(4)]).astype(np.float32)
    K = R.gardner_slope(BETA)
    loop = sdr.tsync_loop_design(0.01, 0.707, K, 4.0) + (2.0, 0.01)
    T = 4 * ONE
    ts = sdr.Tsync(taps, P, T, loop, n_channels=4, stream=st)
    cap = int(ts.max_output(nf).max())
    d_sym = torch.empty((4, cap), dtype=torch.complex64, device=dev)
    d_pos = torch.empty((4, cap, 2), dtype=torch.int64, device=dev)
    d_err = torch.empty((4, cap), dtype=torch.float32, device=dev)
    got = ts.process_dev(d_y, nf, nf, d_sym, cap, cap, d_pos, d_err)
    host = sdr.Tsync(taps, P, T, loop, n_channels=4).process(yh)
    z, po, er = d_sym.cpu().numpy(), d_pos.cpu().numpy().view(np.uint64), d_err.cpu().numpy()
    for k in range(4):
        g = int(got[k])
        assert len(host[0][k]) == g
        assert np.array_equal(_bits(z[k, :g]), _bits(host[0][k])) and np.array_equal(_bits(er[k, :g]),
                                                                                       _bits(host[2][k]))
        pos = [(int(a) << 64) | int(b) for a, b in po[k, :g]]
        assert pos == host[1][k]
        vs, _ = R.replay(pos, er[k, :g], T, _loop_of(loop, 0), first=0)
        d_out = (delays[k] - (D - 1) + (Ld - 1) / 2) / D
        r = R.tracking(pos, z[k, :g], vs, T, 4 * (1 + ppms[k]), d_out, c, ACQ)
        assert r[0] < BAR_TIMING and r[1] < BAR_EVM and abs(r[2]) < BAR_PPM, (k, r)


def test_tsync_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "tsync_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "TSYNC MIRROR OK" in r.stdout, r.stdout + r.stderr

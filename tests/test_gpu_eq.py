"""Adaptive equalizer bank (sdr_eq): every y_s, every e_s and the final taps equal the float32 model (eq_ref.model) bit
for bit at every lane width W, with shared and per-channel adaptation, orders and CMA/DD phases mixed inside warps,
switch points mid-call and mid-tile, random initial taps and inputs scaled by 1e-3 and 1e3; mu = 0 is the fixed FIR;
blind equalisation of BPSK, QPSK and 8PSK on the multipath workload within the model's bars; blockings, clones, resets,
strides, in place and host against device give the same bits; NaN; the launch count; the device-resident
sdr_ddc -> sdr_tsync -> sdr_eq -> sdr_csync chain; the lifecycle of clones; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import csync_ref as CR
import eq_ref as R
import gen
import tsync_ref as TR
from test_csync_host import BAR_EVM, BAR_FREQ, KD
from test_eq_host import BARS, EMAX, ESN0, MU, NSYM, NTAPS, RADIUS, SWITCH, adapt_for, workload_metrics

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _same(a, b):
    """bit for bit, except that any NaN equals any NaN (numpy and the device choose different NaN payloads)"""
    a, b = np.ascontiguousarray(a).view(np.float32), np.ascontiguousarray(b).view(np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32),
                                                                            b[~nb].view(np.uint32))


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n).astype(np.complex64)


def _mixed(C_, n, seed):
    """per-channel adaptation: orders 2, 4, 8 and CMA only, DD only and switches mid-call (37) and mid-tile (150)
    side by side in every warp; inputs and radii scaled by 1, 1e-3 or 1e3 per channel"""
    adapts, scale = [], []
    for k in range(C_):
        sc = [1.0, 1e-3, 1e3][(k // 4) % 3]
        S = [None, 0, 37, 150][k % 4]
        adapts.append(([2, 4, 8][k % 3], [0.01, 0.003, 0.02][(k // 3) % 3] / (sc * sc), sc, 2.0 * sc, S))
        scale.append(sc)
    x = _rows(C_, n, seed) * np.array(scale, np.float32)[:, None]
    return adapts, x.astype(np.complex64)


def _random_taps(C_, N, seed):
    rng = np.random.default_rng(seed)
    t = ((rng.standard_normal((C_, N)) + 1j * rng.standard_normal((C_, N))) * (0.3 / N)).astype(np.complex64)
    t[:, (N - 1) // 2] += 1
    return t


def _check_model(eq, x, N, adapts, taps0, y, e, n=None):
    ym, em, tm = R.model(x, N, adapts, taps0, n)
    for k in range(len(x)):
        nk = x.shape[1] if n is None else int(n[k])
        assert _same(y[k][:nk], ym[k, :nk]), ("y", k, np.nonzero(_bits(y[k][:nk]) != _bits(ym[k, :nk]))[0][:4])
        assert _same(e[k][:nk], em[k, :nk]), ("e", k)
        assert _same(eq.taps(k), tm[k]), ("taps", k)


@pytest.mark.parametrize("C_,N,shared", [(1, 1, True), (3, 2, False), (17, 5, True), (256, 8, False),
                                         (1024, 11, False), (1, 16, True), (3, 31, False), (17, 32, False),
                                         (256, 33, False), (1024, 64, True), (17, 11, True), (1024, 5, False),
                                         (3, 64, False), (256, 16, True)])
def test_eq_bit_exact_against_the_model(sdr, C_, N, shared):
    n = 3 * 32 + 21 if C_ >= 256 else 700
    adapts, x = _mixed(C_, n, C_ + N)
    if shared:
        adapts = (4, 0.01, 1.0, 2.0, 150) if N % 2 else (8, 0.005, 1.0, 1.0, 37)
        x = _rows(C_, n, C_ + N)
    # initial taps: a row per channel, one row shared by every channel (C = 256), or the centre spike
    taps0 = _random_taps(C_, N, N) if C_ % 2 else _random_taps(1, N, N)[0] if C_ == 256 else None
    eq = sdr.Eq(N, adapts, n_channels=C_, taps=taps0)
    y, e = eq.process(x)
    _check_model(eq, x, N, adapts, taps0, y, e)


def test_eq_banks_of_different_tap_counts_side_by_side(sdr):
    """banks whose CTAs need different shared memory (N = 5, 11, 1 and 64: 6592, 3488, 50 688 and 2560 bytes), each
    called again after a bank with another footprint was created: the N = 5 bank after the smaller N = 11 one, the
    N = 1 bank after the smaller N = 64 one.  Every bank's two calls equal the model of its whole stream bit for bit."""
    C_, n = 40, 300
    x = _rows(C_, 2 * n, 77)
    ad = (4, 0.01, 1.0, 2.0, 100)
    out = {}

    def call(N, part):
        y, e = banks[N].process(x[:, part * n:(part + 1) * n])
        out.setdefault(N, []).append((y, e))
    banks = {5: sdr.Eq(5, ad, n_channels=C_)}
    call(5, 0)
    banks[11] = sdr.Eq(11, ad, n_channels=C_)
    call(5, 1)
    call(11, 0)
    banks[1] = sdr.Eq(1, ad, n_channels=C_)
    call(11, 1)
    call(1, 0)
    banks[64] = sdr.Eq(64, ad, n_channels=C_)
    call(1, 1)
    call(64, 0)
    call(64, 1)
    for N, eq in banks.items():
        y = [np.concatenate([out[N][0][0][k], out[N][1][0][k]]) for k in range(C_)]
        e = [np.concatenate([out[N][0][1][k], out[N][1][1][k]]) for k in range(C_)]
        _check_model(eq, x, N, ad, None, y, e)


def test_eq_mu_zero_is_the_fixed_fir(sdr):
    """mu = 0: the model bit for bit and within 1e-6 ||w||_1 max|x| of the f64 convolution; the centre spike gives
    y_s = x_{s-c} bit for bit"""
    for N in (1, 7, 32, 33, 64):
        C_, n = 5, 2000
        x = _rows(C_, n, N)
        t = _random_taps(C_, N, 100 + N)
        eq = sdr.Eq(N, (8, 0.0, 1.0, 2.0, 1000), n_channels=C_, taps=t)
        y, e = eq.process(x)
        _check_model(eq, x, N, (8, 0.0, 1.0, 2.0, 1000), t, y, e)
        for k in range(C_):
            ref = np.convolve(t[k].astype(np.complex128), x[k].astype(np.complex128))[:n]
            bar = 1e-6 * np.abs(t[k]).sum() * np.abs(x[k]).max()
            assert np.abs(y[k] - ref).max() <= bar, (N, k)
            assert np.array_equal(_bits(eq.taps(k)), _bits(t[k]))
        y, _ = sdr.Eq(N, (4, 0.0, 1.0, 2.0, None), n_channels=C_).process(x)
        c = (N - 1) // 2
        for k in range(C_):
            assert np.array_equal(_bits(y[k][c:]), _bits(x[k, :n - c])) and (y[k][:c] == 0).all()


def test_eq_blind_equalisation(sdr):
    """256 channels, BPSK, QPSK and 8PSK with CMA only and with the switch to DD, every order in every warp, on the
    multipath workload: within the model's bars (test_eq_host.py); plus a QPSK channel with a 1e-3 turn-per-symbol
    carrier offset under CMA only, whose ISI bar still holds (CMA is phase-blind)"""
    C_ = 256
    rng = np.random.default_rng(23)
    cases = [(M, S) for S in (None, SWITCH) for M in (2, 4, 8)]
    kinds = [cases[k % 6] for k in range(C_)]
    x = np.empty((C_ + 1, NSYM), np.complex64)
    h = np.empty((C_ + 1, 3), np.complex128)
    a = np.empty((C_ + 1, NSYM + 2), np.complex128)
    for M, S in cases:
        idx = [k for k in range(C_) if kinds[k] == (M, S)]
        x[idx], h[idx], a[idx] = R.multipath_rows(M, len(idx), NSYM, ESN0, rng)
    x[C_:], h[C_:], a[C_:] = R.multipath_rows(4, 1, NSYM, ESN0, rng, freq=[1e-3])
    adapts = [adapt_for(M, S) for M, S in kinds] + [adapt_for(4, None)]
    eq = sdr.Eq(NTAPS, adapts)
    y, _ = eq.process(x)
    y = np.array(y)
    taps = np.array([eq.taps(k) for k in range(C_ + 1)])
    for M, S in cases:
        idx = [k for k in range(C_) if kinds[k] == (M, S)]
        isi, ev = workload_metrics(y[idx], taps[idx], h[idx], a[idx])
        print("M = %d, S = %s: ISI worst %.1f dB, EVM worst %.3f" % (M, S, isi.max(), ev.max()))
        assert isi.max() < BARS[(M, S)][0] and ev.max() < BARS[(M, S)][1], (M, S, isi.max(), ev.max())
    isi_f = R.isi_db(taps[C_], h[C_], 1e-3)
    print("QPSK CMA at 1e-3 turn per symbol: ISI %.1f dB" % isi_f)
    assert isi_f < BARS[(4, None)][0]


def test_eq_blockings_clone_reset_strides_in_place(sdr):
    C_, N, nf = 5, 13, 1500
    adapts, x = _mixed(C_, nf, 9)
    taps0 = _random_taps(C_, N, 10)

    def make(**kw):
        return sdr.Eq(N, adapts, taps=taps0, **kw)

    def same(a, b):
        assert _same(a[0], b[0]) and _same(a[1], b[1])

    def cat(parts, k):
        return tuple(np.concatenate([p[i][k] for p in parts]) for i in range(2))

    one_h = make()
    one = one_h.process(x)
    ref = [(one[0][k], one[1][k]) for k in range(C_)]
    ref_taps = [one_h.taps(k) for k in range(C_)]
    _check_model(one_h, x, N, adapts, taps0, one[0], one[1])
    # 1-symbol calls
    p = make()
    parts = [p.process(x[:, m:m + 1]) for m in range(200)] + [p.process(x[:, 200:])]
    for k in range(C_):
        same(cat(parts, k), ref[k])
        assert _same(p.taps(k), ref_taps[k])
    # random splits, different per channel, with a clone mid-stream
    rng = np.random.default_rng(11)
    p = make()
    at = np.zeros(C_, np.int64)
    parts, clone = [], None
    while (at < nf).any():
        take = np.minimum(nf - at, rng.integers(0, 90, C_))
        parts.append(p.process([x[k, at[k]:at[k] + take[k]] for k in range(C_)]))
        at += take
        if clone is None and at.min() > nf // 2:
            clone, cat_at = p.clone(), at.copy()
    for k in range(C_):
        same(cat(parts, k), ref[k])
    cz = clone.process([x[k, cat_at[k]:] for k in range(C_)])
    for k in range(C_):
        same((cz[0][k], cz[1][k]), tuple(r[cat_at[k]:] for r in ref[k]))
        assert _same(clone.taps(k), ref_taps[k])
    p.reset()
    assert np.array_equal(_bits(p.taps(1)), _bits(taps0[1]))
    again = p.process(x)
    for k in range(C_):
        same((again[0][k], again[1][k]), ref[k])
    # odd device strides give the host bits, and nothing past the counts is written
    torch, dev = _torch()
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = x
    d_x = torch.from_numpy(pad).to(dev)
    q = make(stream=st)
    d_y = torch.full((C_, nf + 3), float("nan"), dtype=torch.complex64, device=dev)
    d_e = torch.full((C_, nf + 3), float("nan"), dtype=torch.complex64, device=dev)
    q.process_dev(d_x, nf, nf + 5, d_y, nf + 3, d_e)
    out, er = d_y.cpu().numpy(), d_e.cpu().numpy()
    for k in range(C_):
        same((out[k, :nf], er[k, :nf]), ref[k])
        assert np.isnan(out[k, nf:]).all() and np.isnan(er[k, nf:]).all()
    # in place on the device, with ragged counts and e not asked for
    q = make(stream=st)
    n = np.array([nf, 1, 0, 777, nf - 1])
    q.process_dev(d_x, n, nf + 5, d_x, nf + 5)
    got = d_x.cpu().numpy()
    for k in range(C_):
        assert _same(got[k, :n[k]], ref[k][0][:n[k]]), k
        assert np.array_equal(_bits(got[k, n[k]:nf]), _bits(x[k, n[k]:])), k
    # in place on the host; different strides for the same rows are refused
    y = x.copy()
    nn = np.full(C_, nf, np.uintp)
    h = make()
    assert sdr.lib().sdr_eq_process(h.h, y.ctypes.data, nn.ctypes.data, nf, y.ctypes.data, None, nf) == 0
    for k in range(C_):
        assert _same(y[k], ref[k][0]), k
    h = make()
    assert sdr.lib().sdr_eq_process(h.h, y.ctypes.data, nn.ctypes.data, nf, y.ctypes.data, None, nf + 1) == 100
    # misaligned device pointers are refused before anything runs
    rc = sdr.lib().sdr_eq_process_dev(h.h, d_x.data_ptr() + 4, nn.ctypes.data, nf + 5, d_y.data_ptr(), None, nf + 3)
    assert rc == 105 and np.array_equal(_bits(h.taps(0)), _bits(taps0[0]))


def test_eq_host_call_larger_than_the_chunk(sdr):
    """one host call of more symbols than the host path moves per round gives process_dev's bits"""
    torch, dev = _torch()
    C_, N = 2, 33
    nf = (1 << 21) + 777  # the host path moves 2^21 symbols per channel per round at C = 2
    adapts = [(4, 0.003, 1.0, 2.0, 1 << 20), (8, 0.002, 1.0, 2.0, None)]
    x = _rows(C_, nf, 13)
    hh = sdr.Eq(N, adapts)
    host = hh.process(x)
    st = torch.cuda.current_stream(dev)
    b = sdr.Eq(N, adapts, stream=st)
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.empty_like(d_x)
    d_e = torch.empty_like(d_x)
    b.process_dev(d_x, nf, nf, d_y, nf, d_e)
    y, e = d_y.cpu().numpy(), d_e.cpu().numpy()
    for k in range(C_):
        assert _same(host[0][k], y[k]) and _same(host[1][k], e[k]) and _same(hh.taps(k), b.taps(k))
    del d_x, d_y, d_e


def test_eq_nan(sdr):
    """a NaN or Inf symbol makes exactly the N outputs whose delay line holds it non-finite, with e = 0 and the taps
    unchanged across them; the outputs before it are those of the clean run bit for bit, and the model still matches"""
    C_, N, nf, m = 3, 7, 2000, 1234
    adapts = [(4, 0.01, 1.0, 2.0, None), (8, 0.01, 1.0, 2.0, 500), (2, 0.01, 1.0, 2.0, 0)]
    x = _rows(C_, nf, 21)
    bad = x.copy()
    bad[1, m] = complex(np.nan, 0.0)
    bad[2, m] = complex(1.0, np.inf)
    eq = sdr.Eq(N, adapts)
    y, e = eq.process(bad)
    _check_model(eq, bad, N, adapts, None, y, e)
    ref, _ = sdr.Eq(N, adapts).process(x)
    assert np.array_equal(_bits(y[0]), _bits(ref[0]))
    for k in (1, 2):
        assert np.array_equal(_bits(y[k][:m]), _bits(ref[k][:m]))
        assert not np.isfinite(y[k][m:m + N]).any() and (e[k][m:m + N] == 0).all()
        assert np.isfinite(y[k][m + N:]).all() and np.isfinite(e[k]).all()
        before, after = sdr.Eq(N, adapts), sdr.Eq(N, adapts)
        before.process(bad[:, :m])
        after.process(bad[:, :m + N])
        assert np.array_equal(_bits(before.taps(k)), _bits(after.taps(k)))


@pytest.mark.parametrize("C_", [1, 1024])
def test_eq_launch_count(sdr, C_):
    torch, dev = _torch()
    b = sdr.Eq(NTAPS, (4, MU, RADIUS, EMAX, SWITCH), n_channels=C_)
    n = 2000
    d_x = torch.randn((C_, n), dtype=torch.complex64, device=dev)
    d_y = torch.empty_like(d_x)
    before = sdr.kernel_launch_count()
    b.process_dev(d_x, n, n, d_y, n)
    assert sdr.kernel_launch_count() - before == 1
    torch.cuda.synchronize()


def test_ddc_to_tsync_to_eq_to_csync_chain(sdr):
    """four RRC QPSK channels (64 input samples per symbol, random carrier phases), each with a symbol-spaced echo
    pair (0.4 one symbol late and 0.25 one symbol early, random phases), in one u8 IQ capture; sdr_ddc is mistuned to
    residual carriers of 0, +1e-3, -2e-3 and 0 turn per symbol -> sdr_ddc (u8, tensor path, D = 16) -> sdr_tsync at 4
    frames per symbol -> sdr_eq (CMA, N = 11, a = 1) -> sdr_csync (QPSK, designed for the equalizer's radius, with no
    measured amplitude; sdr_tsync's matched filter is still scaled by the measured power of the sdr_ddc output, as in
    test_gpu_csync.py, so only the carrier loop's design is free of measurement), device-resident: equal to the host-hop chain bit for bit; after acquisition csync's EVM and
    frequency bars hold.  The same chain without sdr_eq misses the EVM bar on every channel.  csync's RMS phase bar is
    not applied: a CMA equalizer leaves its output at an arbitrary phase, so the carrier phase the loop must follow is
    not the capture's."""
    torch, dev = _torch()
    n, D, Ld, sps = 1 << 22, 16, 255, 64
    freqs = [0.1, -0.27, 0.3, -0.05]
    resid = [0.0, 1e-3, -2e-3, 0.0]
    rng = np.random.default_rng(43)
    x = np.zeros(n, np.complex128)
    for f in freqs:
        s, _ = TR.qpsk_channel(n, sps, rng.uniform(0, sps), 0.35, 8, 80.0, rng)
        s = s.astype(np.complex128)
        ph = np.exp(2j * np.pi * rng.uniform(0, 1, 2))
        s = s + 0.4 * ph[0] * np.roll(s, sps) + 0.25 * ph[1] * np.roll(s, -sps)
        s /= np.sqrt(1 + 0.4 ** 2 + 0.25 ** 2)
        x += s * np.exp(2j * np.pi * (f * np.arange(n) + rng.uniform()))
    raw = np.empty(2 * n, np.uint8)
    raw[0::2] = np.clip(np.round(128 + 12 * x.real), 0, 255)
    raw[1::2] = np.clip(np.round(128 + 12 * x.imag), 0, 255)
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0)
    st = torch.cuda.current_stream(dev)
    ddc = sdr.Ddc(hd, [f - r / sps for f, r in zip(freqs, resid)], 1.0, D, "u8iq", stream=st)
    nf = n // D
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((4, nf), dtype=torch.complex64, device=dev)
    assert ddc.process_dev(d_in, n, d_y, nf, nf) == nf
    yh = d_y.cpu().numpy()
    P = 32
    h, _ = TR.rrc_taps(4.0, P, 0.35, 8)
    taps = np.stack([h / np.sqrt((np.abs(yh[k]) ** 2).mean()) for k in range(4)]).astype(np.float32)
    tloop = sdr.tsync_loop_design(0.01, 0.707, TR.gardner_slope(0.35), 4.0) + (2.0, 0.01)
    ts = sdr.Tsync(taps, P, 4 << 64, tloop, n_channels=4, stream=st)
    cap = int(ts.max_output(nf).max())
    d_sym = torch.empty((4, cap), dtype=torch.complex64, device=dev)
    got = ts.process_dev(d_y, nf, nf, d_sym, cap, cap)
    eadapt = (4, MU, RADIUS, EMAX, None)
    eq = sdr.Eq(NTAPS, eadapt, n_channels=4, stream=st)
    d_q = torch.empty_like(d_sym)
    eq.process_dev(d_sym, got, cap, d_q, cap)
    # the loop is designed for the equalizer's radius: no amplitude is measured
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, KD[4] * RADIUS, 1 / (2 * np.pi))
    loop = (4, kp, ki, 2.0 * RADIUS, 0.02)
    cs = sdr.Csync(loop, n_channels=4, stream=st)
    d_z = torch.empty_like(d_sym)
    d_ph = torch.empty((4, cap), dtype=torch.int64, device=dev)
    d_e = torch.empty((4, cap), dtype=torch.float32, device=dev)
    cs.process_dev(d_q, got, cap, d_z, cap, d_ph, d_e)
    z, po, er = d_z.cpu().numpy(), d_ph.cpu().numpy().view(np.uint64), d_e.cpu().numpy()
    hs = sdr.Tsync(taps, P, 4 << 64, tloop, n_channels=4).process(yh)[0]
    hq = sdr.Eq(NTAPS, eadapt, n_channels=4).process(hs)[0]
    host = sdr.Csync(loop, n_channels=4).process(hq)
    without = sdr.Csync(loop, n_channels=4).process(hs)
    skip = 20000
    for k in range(4):
        g = int(got[k])
        assert len(hs[k]) == g and g > skip + 10000
        assert np.array_equal(_bits(z[k, :g]), _bits(host[0][k])) and np.array_equal(po[k, :g], host[1][k])
        assert np.array_equal(_bits(er[k, :g]), _bits(host[2][k]))
        nus, _ = CR.replay([po[k, :g]], [er[k, :g]], [g], loop, 0, 0)
        _, evm, df = CR.tracking(4, z[None, k, :g], po[None, k, :g], nus, np.zeros(1), [resid[k]], skip)
        nus_w, _ = CR.replay([without[1][k]], [without[2][k]], [g], loop, 0, 0)
        _, evm_w, _ = CR.tracking(4, without[0][k][None], without[1][k][None], nus_w, np.zeros(1), [resid[k]], skip)
        print("channel %d: EVM %.4f with sdr_eq, %.4f without; |nu - f| %.3g" % (k, evm[0], evm_w[0], df[0]))
        assert df[0] < BAR_FREQ and evm[0] < BAR_EVM, (k, df, evm)
        assert evm_w[0] > BAR_EVM, (k, evm_w)


def _lifecycle_blocks():
    rows = _rows(2, 6000, 31)
    return np.split(rows, [2345], axis=1)


@pytest.mark.parametrize("caller_stream", [False, True], ids=["own_stream", "caller_stream"])
def test_eq_clone_outlives_its_source(sdr, caller_stream):
    """as test_gpu_handle_lifecycle.py for the other handles: process a block, clone, close the source, finish on the
    clone: the bits of a fresh handle fed the same blocks, and a caller stream still takes work afterwards"""
    import torch
    st = torch.cuda.Stream() if caller_stream else None
    bs = _lifecycle_blocks()
    adapts = [(4, 0.01, 1.0, 2.0, 3000), (8, 0.01, 1.0, 2.0, None)]

    def run(h, b):
        y, e = h.process(np.ascontiguousarray(b))
        return [y[0], y[1], e[0], e[1], h.taps(0), h.taps(1)]
    fresh = sdr.Eq(NTAPS, adapts, stream=st)
    run(fresh, bs[0])
    want = run(fresh, bs[1])
    fresh.close()
    src = sdr.Eq(NTAPS, adapts, stream=st)
    run(src, bs[0])
    clone = src.clone()
    src.close()
    got = run(clone, bs[1])
    clone.close()
    for g, w in zip(got, want):
        assert np.array_equal(_bits(g), _bits(w))
    if caller_stream:
        with torch.cuda.stream(st):
            t = torch.arange(4096, device="cuda", dtype=torch.float32) * 2.0
        st.synchronize()
        assert t.sum().item() == 4095.0 * 4096.0


def test_eq_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "eq_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "EQ MIRROR OK" in r.stdout, r.stdout + r.stderr

"""Carrier recovery bank (sdr_csync): the loop's integer recurrence replayed exactly from the reported errors; every error
equal to the float32 detector of its reported symbol bit for bit; every symbol against the f64 rotation at its exact
phase; the open loop; acquisition and tracking of BPSK, QPSK and 8PSK at known offsets and phases, and saturation of
nu at +-V; blockings, clones, resets, strides, in place and host against device give the same bits; NaN; the launch
count; the device-resident sdr_ddc -> sdr_tsync -> sdr_csync chain; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import csync_ref as R
import gen
import tsync_ref as TR
from test_csync_host import ACQ, BAR_EVM, BAR_FREQ, BAR_PHASE, ESN0, KD, N, OFFSETS, design

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
ROT_BAR = 1e-6  # |z - x e^{-2 pi i phi / 2^64}| / |x|

# valid loops of every order with corrections large enough that the errors steer the phase visibly
LOOPS = [(4, 0.004, 3e-5, 2.0, 0.01), (2, 0.02, 5e-4, 1.0, 0.05), (8, 0.01, 1e-4, 1.5, 1 / 16), (4, 0.0, 0.0, 1.0, 0.0),
         (8, 0.003, 2e-5, 2.0, 0.001), (2, 0.1, 0.01, 2.0, 0.25)]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n)


def _loop_list(loops, C_):
    return [loops] * C_ if np.ndim(loops[0]) == 0 else list(loops)


def _start(C_, loops, seed):
    """phi_0 random, at 2^63 (f = -1/2) and 0; nu_0 nonzero within each channel's V"""
    rng = np.random.default_rng(seed)
    lp = _loop_list(loops, C_)
    phi0 = [[int(rng.integers(0, 1 << 63)) * 2 + 1, 1 << 63, 0][k % 3] for k in range(C_)]
    nu0 = [int(rng.integers(-R.dev_bound(lp[k][4]), R.dev_bound(lp[k][4]) + 1)) for k in range(C_)]
    return phi0, nu0


def _check_exact(cs, x, n, loops, phi0, nu0, z, ph, err):
    """replay of every phase and the final state; errors equal the f32 detector of z bit for bit; z against f64"""
    C_ = len(z)
    lp = _loop_list(loops, C_)
    _, (phi_n, nu_n) = R.replay(ph, err, n, loops, phi0, nu0)
    worst = 0.0
    for k in range(C_):
        assert cs.state(k) == (int(phi_n[k]), int(nu_n[k])), k
        zk = np.asarray(z[k], np.complex64)
        g = R.detector(zk.real, zk.imag, lp[k][0])
        assert np.array_equal(_bits(R.clamp_err(g, lp[k][3])), _bits(err[k])), k
        xk = np.asarray(x[k][:n[k]], np.complex128)
        d = np.abs(zk - R.rotate(xk, ph[k])) / np.abs(xk)
        worst = max(worst, float(d.max(initial=0)))
    assert worst <= ROT_BAR, worst
    return worst


@pytest.mark.parametrize("C_,shared,M", [(1, True, 4), (1, True, 8), (3, False, None), (17, True, 2),
                                         (17, False, None), (256, True, 8), (256, False, None), (1024, True, 4),
                                         (1024, False, None)])
def test_csync_exact_loop_arithmetic(sdr, C_, shared, M):
    loops = next(lp for lp in LOOPS if lp[0] == M) if shared else [LOOPS[k % len(LOOPS)] for k in range(C_)]
    phi0, nu0 = _start(C_, loops, C_)
    nf = 3000 if C_ <= 17 else 500
    x = _rows(C_, nf, C_ + 1) * 2
    cs = sdr.Csync(loops, n_channels=C_, phase=phi0, freq=nu0)
    z, ph, err = cs.process(x)
    worst = _check_exact(cs, x, [nf] * C_, loops, phi0, nu0, z, ph, err)
    print("worst |z - x r| / |x| = %.3g" % worst)


def test_csync_open_loop(sdr):
    """kp = ki = 0: phi_s = phi_0 + s 2^24 nu_0 exactly; phi_0 = nu_0 = 0: z = x bit for bit"""
    C_, nf = 5, 2000
    x = _rows(C_, nf, 2)
    phi0 = [0, 1 << 63, 12345, (1 << 64) - 1, 1 << 62]
    nu0 = [0, R.dev_bound(0.01), -R.dev_bound(0.01), 7, -(1 << 30)]
    cs = sdr.Csync((4, 0.0, 0.0, 1.0, 0.01), phase=phi0, freq=nu0)
    z, ph, err = cs.process(x)
    for k in range(C_):
        assert [int(p) for p in ph[k]] == [(phi0[k] + s * (nu0[k] << 24)) % (1 << 64) for s in range(nf)]
        assert cs.state(k) == ((phi0[k] + nf * (nu0[k] << 24)) % (1 << 64), nu0[k])
        assert np.abs(z[k] - R.rotate(x[k], ph[k])).max() <= ROT_BAR * np.abs(x[k]).max()
    assert np.array_equal(_bits(z[0]), _bits(x[0]))


def test_csync_acquires_and_tracks(sdr):
    """256 channels, orders 2, 4 and 8 side by side in every warp, at the CPU model's offsets, random phases and Es/N0:
    within the model's bars after ACQ symbols (test_csync_host.py)"""
    C_ = 256
    orders = [[2, 4, 8][k % 3] for k in range(C_)]
    offs = [OFFSETS[k % 5] for k in range(C_)]
    rng = np.random.default_rng(7)
    x = np.empty((C_, N), np.complex64)
    theta = np.empty(C_)
    for M in (2, 4, 8):
        idx = [k for k in range(C_) if orders[k] == M]
        x[idx], theta[idx], _ = R.psk_rows(M, [offs[k] for k in idx], N, ESN0, rng)
    loops = [design(sdr, M) for M in orders]
    cs = sdr.Csync(loops)
    z, ph, err = cs.process(x)
    z, ph = np.array(z), np.array(ph)
    nus, (phi_n, nu_n) = R.replay(ph, err, [N] * C_, loops, 0, 0)
    worst = np.zeros(3)
    for M in (2, 4, 8):
        idx = [k for k in range(C_) if orders[k] == M]
        r = R.tracking(M, z[idx], ph[idx], nus[idx], theta[idx], [offs[k] for k in idx], ACQ)
        worst = np.maximum(worst, [a.max() for a in r])
    assert worst[0] < BAR_PHASE and worst[1] < BAR_EVM and worst[2] < BAR_FREQ, worst
    print("worst RMS phase error %.4f rad, EVM %.4f, |nu - f| %.3g turn per symbol" % tuple(worst))


def test_csync_offset_beyond_max_freq_saturates(sdr):
    """+-2e-3 turn per symbol against max_freq = 1e-3: nu never passes V and reaches exactly +-V, the offset's sign"""
    offs = [2e-3, -2e-3, 2e-3, -2e-3]
    rng = np.random.default_rng(8)
    x, _, _ = R.psk_rows(4, offs, N, ESN0, rng)
    loop = design(sdr, 4)[:4] + (1e-3,)
    cs = sdr.Csync(loop, n_channels=4)
    z, ph, err = cs.process(x)
    nus, _ = R.replay(ph, err, [N] * 4, loop, 0, 0)
    V = R.dev_bound(1e-3)
    for k in range(4):
        sign = 1 if offs[k] > 0 else -1
        assert np.abs(nus[k]).max() == V and (nus[k, ACQ:] == sign * V).sum() > (N - ACQ) // 10, k


def test_csync_blockings_clone_reset_strides_in_place(sdr):
    C_, nf = 5, 1500
    loops = [LOOPS[k % len(LOOPS)] for k in range(C_)]
    phi0, nu0 = _start(C_, loops, 9)
    x = _rows(C_, nf, 10) * 2

    def make(**kw):
        return sdr.Csync(loops, phase=phi0, freq=nu0, **kw)

    def same(a, b):
        assert np.array_equal(_bits(a[0]), _bits(b[0])) and np.array_equal(a[1], b[1]) and \
            np.array_equal(_bits(a[2]), _bits(b[2]))

    def cat(parts, k):
        return tuple(np.concatenate([p[i][k] for p in parts]) for i in range(3))

    one = make().process(x)
    ref = [(one[0][k], one[1][k], one[2][k]) for k in range(C_)]
    # 1-symbol calls
    p = make()
    parts = [p.process(x[:, m:m + 1]) for m in range(300)] + [p.process(x[:, 300:])]
    for k in range(C_):
        same(cat(parts, k), ref[k])
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
        same((cz[0][k], cz[1][k], cz[2][k]), tuple(r[cat_at[k]:] for r in ref[k]))
    p.reset()
    assert p.state(1) == (phi0[1], nu0[1])
    again = p.process(x)
    for k in range(C_):
        same((again[0][k], again[1][k], again[2][k]), ref[k])
    # odd device strides give the host bits, and nothing past the counts is written
    torch, dev = _torch()
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = x
    d_x = torch.from_numpy(pad).to(dev)
    q = make(stream=st)
    d_z = torch.full((C_, nf + 3), float("nan"), dtype=torch.complex64, device=dev)
    d_ph = torch.zeros((C_, nf + 3), dtype=torch.int64, device=dev)
    d_e = torch.full((C_, nf + 3), float("nan"), dtype=torch.float32, device=dev)
    q.process_dev(d_x, nf, nf + 5, d_z, nf + 3, d_ph, d_e)
    out, po, er = d_z.cpu().numpy(), d_ph.cpu().numpy().view(np.uint64), d_e.cpu().numpy()
    for k in range(C_):
        same((out[k, :nf], po[k, :nf], er[k, :nf]), ref[k])
        assert np.isnan(out[k, nf:]).all() and np.isnan(er[k, nf:]).all() and (po[k, nf:] == 0).all()
    # in place on the device, with ragged counts and phase / err not asked for
    q = make(stream=st)
    n = np.array([nf, 1, 0, 777, nf - 1])
    q.process_dev(d_x, n, nf + 5, d_x, nf + 5)
    got = d_x.cpu().numpy()
    for k in range(C_):
        assert np.array_equal(_bits(got[k, :n[k]]), _bits(ref[k][0][:n[k]])), k
        assert np.array_equal(_bits(got[k, n[k]:nf]), _bits(x[k, n[k]:])), k
    # in place on the host; different strides for the same rows are refused
    y = x.copy()
    nn = np.full(C_, nf, np.uintp)
    h = make()
    assert sdr.lib().sdr_csync_process(h.h, y.ctypes.data, nn.ctypes.data, nf, y.ctypes.data, None, None, nf) == 0
    for k in range(C_):
        assert np.array_equal(_bits(y[k]), _bits(ref[k][0])), k
    h = make()
    assert sdr.lib().sdr_csync_process(h.h, y.ctypes.data, nn.ctypes.data, nf, y.ctypes.data, None, None,
                                       nf + 1) == 100
    # misaligned device pointers are refused
    rc = sdr.lib().sdr_csync_process_dev(h.h, d_x.data_ptr() + 4, nn.ctypes.data, nf + 5, d_z.data_ptr(), None,
                                         None, nf + 3)
    assert rc == 105 and h.state(0) == (phi0[0], nu0[0])


def test_csync_host_call_larger_than_the_chunk(sdr):
    """one host call of more symbols than the host path moves per round gives process_dev's bits"""
    torch, dev = _torch()
    C_ = 2
    nf = (1 << 21) + 777  # the host path moves 2^21 symbols per channel per round at C = 2
    loops = [LOOPS[0], LOOPS[2]]
    x = _rows(C_, nf, 13) * 2
    host = sdr.Csync(loops, phase=[5, 1 << 63], freq=[100, -100]).process(x)
    st = torch.cuda.current_stream(dev)
    b = sdr.Csync(loops, phase=[5, 1 << 63], freq=[100, -100], stream=st)
    d_x = torch.from_numpy(x).to(dev)
    d_z = torch.empty_like(d_x)
    d_ph = torch.empty((C_, nf), dtype=torch.int64, device=dev)
    d_e = torch.empty((C_, nf), dtype=torch.float32, device=dev)
    b.process_dev(d_x, nf, nf, d_z, nf, d_ph, d_e)
    z, po, er = d_z.cpu().numpy(), d_ph.cpu().numpy().view(np.uint64), d_e.cpu().numpy()
    for k in range(C_):
        assert np.array_equal(_bits(host[0][k]), _bits(z[k])) and np.array_equal(host[1][k], po[k])
        assert np.array_equal(_bits(host[2][k]), _bits(er[k]))
    del d_x, d_z, d_ph, d_e


def test_csync_nan(sdr):
    """a NaN symbol gets e = 0 and a NaN z; the symbols before it are those of the NaN-free run bit for bit, and replay
    holds throughout"""
    C_, nf, m = 3, 2000, 1234
    loops = LOOPS[:3]
    phi0, nu0 = _start(C_, loops, 20)
    x = _rows(C_, nf, 21) * 2
    bad = x.copy()
    bad[1, m] = np.complex64(complex(np.nan, 0.0))
    bad[2, m] = np.complex64(complex(1.0, np.inf))
    z, ph, err = sdr.Csync(loops, phase=phi0, freq=nu0).process(bad)
    ref = sdr.Csync(loops, phase=phi0, freq=nu0).process(x)
    R.replay(ph, err, [nf] * C_, loops, phi0, nu0)
    assert np.array_equal(_bits(z[0]), _bits(ref[0][0]))
    for k in (1, 2):
        assert err[k][m] == 0 and not np.isfinite(z[k][m]).all()
        assert np.isfinite(z[k][:m]).all() and np.isfinite(z[k][m + 1:]).all() and np.isfinite(err[k]).all()
        assert np.array_equal(_bits(z[k][:m]), _bits(ref[0][k][:m])) and np.array_equal(ph[k][:m + 1],
                                                                                       ref[1][k][:m + 1])


@pytest.mark.parametrize("C_", [1, 1024])
def test_csync_launch_count(sdr, C_):
    torch, dev = _torch()
    b = sdr.Csync(LOOPS[0], n_channels=C_)
    n = 2000
    d_x = torch.randn((C_, n), dtype=torch.complex64, device=dev)
    d_z = torch.empty_like(d_x)
    before = sdr.kernel_launch_count()
    b.process_dev(d_x, n, n, d_z, n)
    assert sdr.kernel_launch_count() - before == 1
    torch.cuda.synchronize()


def test_ddc_to_tsync_to_csync_chain(sdr):
    """four RRC QPSK channels (64 input samples per symbol, random carrier phases) in one u8 IQ capture; sdr_ddc is
    mistuned so that the residual carriers are 0, +1e-3, -2e-3 and 1e-2 turn per symbol (the last with nu_0 seeded
    7e-4 below it) -> sdr_ddc (u8, tensor path, D = 16) -> sdr_tsync at 4 frames per symbol -> sdr_csync (QPSK) with
    sdr_tsync's counts as n_in, device-resident: equal to the host-hop chain bit for bit; after the acquisitions the
    model's tracking bars hold: the frequency against the residual, the EVM after a real gain fit, and the RMS phase
    error against the carrier theta + resid s with the constant theta fitted modulo a quarter turn"""
    torch, dev = _torch()
    n, D, Ld, sps = 1 << 22, 16, 255, 64
    freqs = [0.1, -0.27, 0.3, -0.05]
    resid = [0.0, 1e-3, -2e-3, 1e-2]
    rng = np.random.default_rng(41)
    x = np.zeros(n, np.complex128)
    for f in freqs:
        s, _ = TR.qpsk_channel(n, sps, rng.uniform(0, sps), 0.35, 8, 80.0, rng)
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
    # the loop is designed for the symbols' amplitude (there is no AGC)
    A = float(np.abs(d_sym.cpu().numpy()[:, 2000:int(got.min())]).mean())
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, KD[4] * A, 1 / (2 * np.pi))
    loop = (4, kp, ki, 2.0 * A, 0.02)
    nu0 = [0, 0, 0, R.dev_bound(1e-2 - 7e-4)]
    cs = sdr.Csync(loop, n_channels=4, freq=nu0, stream=st)
    d_z = torch.empty_like(d_sym)
    d_ph = torch.empty((4, cap), dtype=torch.int64, device=dev)
    d_e = torch.empty((4, cap), dtype=torch.float32, device=dev)
    cs.process_dev(d_sym, got, cap, d_z, cap, d_ph, d_e)
    z, po, er = d_z.cpu().numpy(), d_ph.cpu().numpy().view(np.uint64), d_e.cpu().numpy()
    hs = sdr.Tsync(taps, P, 4 << 64, tloop, n_channels=4).process(yh)[0]
    host = sdr.Csync(loop, n_channels=4, freq=nu0).process(hs)
    skip = 4000
    for k in range(4):
        g = int(got[k])
        assert len(hs[k]) == g and g > skip + 10000
        assert np.array_equal(_bits(z[k, :g]), _bits(host[0][k])) and np.array_equal(po[k, :g], host[1][k])
        assert np.array_equal(_bits(er[k, :g]), _bits(host[2][k]))
        nus, _ = R.replay([po[k, :g]], [er[k, :g]], [g], loop, 0, nu0[k])
        # the carrier at symbol s is theta + resid s; theta (after the DDC's and sdr_tsync's filters) is fitted, modulo
        # a quarter turn, from the phases after acquisition
        t = po[k, skip:g].view(np.int64) * R.TURN_PHI - resid[k] * np.arange(skip, g)
        theta = np.angle(np.exp(2j * np.pi * 4 * t).mean()) / (2 * np.pi * 4)
        rms, evm, df = R.tracking(4, z[None, k, :g], po[None, k, :g], nus, np.array([theta]), [resid[k]], skip)
        assert df[0] < BAR_FREQ and evm[0] < BAR_EVM and rms[0] < BAR_PHASE, (k, df, evm, rms)


def test_csync_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "csync_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "CSYNC MIRROR OK" in r.stdout, r.stdout + r.stderr

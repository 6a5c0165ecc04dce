"""Viterbi decoder bank (sdr_vit): released bits and counts equal the model (vit_ref) bit for bit for K = 3..9,
n = 2..4, L in {32, 64, 96, 512}, C in {1, 3, 17, 256, 1024}, shared and per-channel scales, both start modes and soft
values with saturating, NaN and Inf entries; finish with and without termination and on a subset; one-step calls,
random per-channel splits, calls ending mid-block, clones, resets, host calls larger than the host chunk and host
against device give the same bits; a stream whose least exact metric passes 2^32 equals the C++ model; one launch per
call without a synchronise; BER at scale within the model's bars; clones outlive their source; the C++ mirror; the
sdr_ddc -> sdr_tsync -> sdr_eq -> sdr_csync -> sdr_vit chain."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import gen
import tsync_ref as TR
import vit_ref as R
from test_eq_host import EMAX, MU, NTAPS, RADIUS
from test_csync_host import KD
from test_vit_host import BER_BARS, BER_L, BER_SCALE, _cpp_model, ber_workload, run_cpp_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def soft(C_, steps, K, gens, seed, uniform=False):
    """coded random messages at a moderate SNR, with about 1 % saturating (+-1e30), 0.5 % NaN and 0.5 % +-Inf"""
    rng = np.random.default_rng(seed)
    msg = rng.integers(0, 2, (C_, steps))
    state = rng.integers(0, 1 << (K - 1), C_) if uniform else 0
    x = R.bpsk(R.encode(msg, K, gens, state), 2.0, 1.0 / len(gens), rng)
    u = rng.random(x.shape)
    x[u < 0.01] = np.float32(1e30) * np.sign(rng.standard_normal(int((u < 0.01).sum()))).astype(np.float32)
    x[(u >= 0.01) & (u < 0.015)] = np.nan
    x[(u >= 0.015) & (u < 0.02)] = np.inf * np.sign(rng.standard_normal(int(((u >= 0.015) & (u < 0.02)).sum())))
    return x.astype(np.float32)


# four generators per K; a rate-1/n test uses the first n
CODES = {3: (0o5, 0o7, 0o3, 0o6), 4: (0o15, 0o17, 0o13, 0o11), 5: (0o23, 0o35, 0o33, 0o37), 6: (0o53, 0o75, 0o47, 0o65),
         7: (0o133, 0o171, 0o165, 0o117), 8: (0o247, 0o371, 0o345, 0o273), 9: (0o561, 0o753, 0o711, 0o663)}


@pytest.mark.parametrize("C_,K,n,L,shared,zs", [
    (1, 3, 2, 32, True, True), (3, 4, 3, 64, False, False), (17, 5, 4, 96, True, True), (256, 6, 2, 32, False, True),
    (1024, 7, 2, 64, True, False), (3, 7, 3, 512, False, True), (17, 8, 3, 64, False, False), (1, 9, 2, 96, True, True),
    (256, 9, 4, 32, True, False), (17, 3, 4, 512, False, False), (1024, 5, 2, 32, False, True),
    (3, 9, 3, 512, True, False), (1024, 9, 2, 64, False, True), (256, 4, 2, 96, True, True)])
def test_vit_bit_exact_against_the_model(sdr, C_, K, n, L, shared, zs):
    g = CODES[K][:n]
    steps = L + 32 + (100 if C_ >= 256 else 413)
    x = soft(C_, steps, K, g, C_ * 100 + K * 10 + n, uniform=not zs)
    scale = np.float32(40.0) if shared else np.linspace(5, 80, C_).astype(np.float32)
    v = sdr.Vit(K, g, L, scale, n_channels=C_, zero_start=zs)
    m = R.Vit(K, g, L, scale, zs, C=C_)
    got = v.process(x)
    want = m.process(x)
    for k in range(C_):
        assert np.array_equal(got[k], want[k]), (k, len(got[k]), len(want[k]))
    which = np.arange(C_) % 2 == 0
    for term in (True, False):
        f = v.finish(which, terminated=term)
        fw = m.finish(which, terminated=term)
        for k in range(C_):
            assert np.array_equal(f[k], fw[k]), ("finish", term, k)
        which = ~which


def test_vit_blockings_finish_clone_reset_host_device(sdr):
    C_, K, L = 5, 7, 64
    g = (0o133, 0o171)
    nf = 1500
    x = soft(C_, nf, K, g, 9)
    scale = [10.0, 20.0, 30.0, 40.0, 50.0]
    mdl = R.Vit(K, g, L, scale, True)
    mid = 777
    ref = [list(b) for b in mdl.process(x[:, :mid])]
    # a finish on a subset mid-stream: listed channels restart from their creation state
    which = np.array([1, 0, 1, 0, 0], bool)
    fin1 = mdl.finish(which, terminated=False)
    rest = mdl.process(x[:, mid:])
    fin2 = mdl.finish(terminated=True)
    want = [np.concatenate([ref[k], fin1[k], rest[k], fin2[k]]).astype(np.uint8) for k in range(C_)]

    def feed(v, parts_fn):
        out = [[] for _ in range(C_)]
        for part in parts_fn(0, mid):
            for k, b in enumerate(v.process(part)):
                out[k].append(b)
        for k, b in enumerate(v.finish(which, terminated=False)):
            out[k].append(b)
        for part in parts_fn(mid, nf):
            for k, b in enumerate(v.process(part)):
                out[k].append(b)
        for k, b in enumerate(v.finish(terminated=True)):
            out[k].append(b)
        return [np.concatenate(o).astype(np.uint8) for o in out]

    def check(got):
        for k in range(C_):
            assert np.array_equal(got[k], want[k]), k

    check(feed(sdr.Vit(K, g, L, scale), lambda a, b: [x[:, a:b]]))
    # one-step calls
    check(feed(sdr.Vit(K, g, L, scale), lambda a, b: [x[:, t:t + 1] for t in range(a, b)]))
    # random per-channel splits, calls ending mid-block
    rng = np.random.default_rng(3)

    def ragged(a, b):
        at = np.full(C_, a)
        while (at < b).any():
            take = np.minimum(b - at, rng.integers(0, 70, C_))
            yield [x[k, at[k]:at[k] + take[k]] for k in range(C_)]
            at += take
    check(feed(sdr.Vit(K, g, L, scale), ragged))
    # clone mid-stream; the clone continues alone
    v = sdr.Vit(K, g, L, scale)
    head = v.process(x[:, :500])
    c = v.clone()
    v.process(x[:, 500:600])
    tail = c.process(x[:, 500:mid])
    for k in range(C_):
        assert np.array_equal(np.concatenate([head[k], tail[k]]), np.asarray(ref[k], np.uint8))
    # reset
    v.reset()
    check(feed(v, lambda a, b: [x[:, a:b]]))
    # the device path with odd strides equals the host path; nothing past the counts is written
    torch, dev = _torch()
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5, 2), np.nan, np.float32)
    pad[:, :nf] = x.reshape(C_, nf, 2)
    d_x = torch.from_numpy(pad).to(dev)
    ostride = 1600
    d_y = torch.full((C_, ostride), 7, dtype=torch.uint8, device=dev)
    d = sdr.Vit(K, g, L, scale, stream=st)
    cnt = d.process_dev(d_x, nf, nf + 5, d_y, ostride)
    y = d_y.cpu().numpy()
    one = sdr.Vit(K, g, L, scale).process(x)
    for k in range(C_):
        assert cnt[k] == len(one[k]) == R.released(nf, L)
        assert np.array_equal(y[k, :cnt[k]], one[k]) and (y[k, cnt[k]:] == 7).all()
    d_f = torch.full((C_, 128), 7, dtype=torch.uint8, device=dev)
    fc = d.finish_dev(d_f, 128, which, terminated=False)
    hv = sdr.Vit(K, g, L, scale)
    hv.process(x)
    hf = hv.finish(which, terminated=False)
    fy = d_f.cpu().numpy()
    for k in range(C_):
        assert fc[k] == len(hf[k]) and np.array_equal(fy[k, :fc[k]], hf[k]) and (fy[k, fc[k]:] == 7).all()
    # misaligned device rows are refused before anything runs
    n = np.full(C_, 64, np.uintp)
    o = np.zeros(C_, np.uintp)
    assert sdr.lib().sdr_vit_process_dev(d.h, d_x.data_ptr(), n.ctypes.data, nf + 5, d_y.data_ptr() + 1, ostride,
                                         o.ctypes.data) == 105
    assert sdr.lib().sdr_vit_process_dev(d.h, d_x.data_ptr(), n.ctypes.data, nf + 5, d_y.data_ptr(), ostride - 2,
                                         o.ctypes.data) == 105


def test_vit_host_call_larger_than_the_chunk(sdr):
    """one host call of more steps than the host path moves per round gives process_dev's bits"""
    torch, dev = _torch()
    C_, K, L = 2, 7, 96
    g = (0o133, 0o171)
    nf = (1 << 21) + 777  # the host path moves 2^21 steps per channel per round at C = 2, n = 2
    x = np.random.default_rng(13).standard_normal((C_, nf, 2)).astype(np.float32)
    host = sdr.Vit(K, g, L, [20.0, 30.0]).process(x)
    st = torch.cuda.current_stream(dev)
    b = sdr.Vit(K, g, L, [20.0, 30.0], stream=st)
    d_x = torch.from_numpy(x).to(dev)
    ostride = (nf + 3) // 4 * 4  # device rows are 4-byte aligned
    d_y = torch.empty((C_, ostride), dtype=torch.uint8, device=dev)
    cnt = b.process_dev(d_x, nf, nf, d_y, ostride)
    y = d_y.cpu().numpy()
    for k in range(C_):
        assert cnt[k] == R.released(nf, L) and np.array_equal(host[k], y[k, :cnt[k]])
    # and the first 4000 steps against the model
    m = R.model(x[:, :4000], K, g, L, [20.0, 30.0], True)
    for k in range(C_):
        assert np.array_equal(host[k][:len(m[k])], m[k])


def test_vit_metric_width(sdr):
    """one n = 4 stream long enough that the model's least exact metric passes 2^32 (mostly erasures, which cost 508
    per step on every path, with random saturated steps between them): equal to the C++ model bit for bit, so a 32-bit
    absolute metric would have wrapped"""
    K, g, L = 5, (0o23, 0o35, 0o33, 0o37), 64
    steps = 10_000_000
    rng = np.random.default_rng(77)
    x = np.zeros((steps, 4), np.float32)
    live = rng.random(steps) < 0.1
    x[live] = rng.choice(np.array([-3.0, 3.0, 0.4, -0.4], np.float32), (int(live.sum()), 4))
    with tempfile.TemporaryDirectory() as tmp:
        want, least = run_cpp_model(_cpp_model(tmp), x, K, g, L, 50.0, True, tmp)
    assert least > 1 << 32
    got = sdr.Vit(K, g, L, 50.0).process(x.reshape(1, -1))[0]
    assert len(got) == len(want) and np.array_equal(got, want)


@pytest.mark.parametrize("C_", [1, 1024])
def test_vit_launch_count_and_no_synchronise(sdr, C_):
    torch, dev = _torch()
    st = torch.cuda.Stream(dev)
    b = sdr.Vit(7, (0o133, 0o171), 64, 20.0, n_channels=C_, stream=st)
    n = 2000
    d_x = torch.randn((C_, n, 2), dtype=torch.float32, device=dev)
    d_y = torch.empty((C_, n), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        torch.cuda._sleep(200_000_000)  # about 0.1 s of device time queued before the call
    before = sdr.kernel_launch_count()
    cnt = b.process_dev(d_x, n, n, d_y, n)
    assert not st.query(), "process_dev waited for the stream"
    assert sdr.kernel_launch_count() - before == 1
    assert (cnt == R.released(n, 64)).all()
    st.synchronize()


def test_vit_ber_at_scale(sdr):
    """256 channels at Eb/N0 = 3 dB stay within the CPU model's bar"""
    K, g = R.CODES["k7"]
    msg, x = ber_workload(3.0, 256, 303)
    v = sdr.Vit(K, g, BER_L, BER_SCALE, n_channels=256)
    b = v.process(x)
    f = v.finish()
    out = np.array([np.concatenate([b[k], f[k]]) for k in range(256)])
    ber = (out != msg).mean()
    print("BER at 3 dB over %d bits: %.3g" % (msg.size, ber))
    assert ber < BER_BARS[3.0]


@pytest.mark.parametrize("caller_stream", [False, True], ids=["own_stream", "caller_stream"])
def test_vit_clone_outlives_its_source(sdr, caller_stream):
    import torch
    st = torch.cuda.Stream() if caller_stream else None
    K, g = R.CODES["k9n3"]
    x = soft(2, 3000, K, g, 31)
    bs = [x[:, :1234], x[:, 1234:]]

    def run(h, blk):
        return h.process(np.ascontiguousarray(blk))
    fresh = sdr.Vit(K, g, 96, 25.0, n_channels=2, stream=st)
    run(fresh, bs[0])
    want = run(fresh, bs[1]) + fresh.finish(terminated=False)
    fresh.close()
    src = sdr.Vit(K, g, 96, 25.0, n_channels=2, stream=st)
    run(src, bs[0])
    clone = src.clone()
    src.close()
    got = run(clone, bs[1]) + clone.finish(terminated=False)
    clone.close()
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    if caller_stream:
        with torch.cuda.stream(st):
            t = torch.arange(4096, device="cuda", dtype=torch.float32) * 2.0
        st.synchronize()
        assert t.sum().item() == 4095.0 * 4096.0


def test_vit_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "vit_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "VIT MIRROR OK" in r.stdout, r.stdout + r.stderr


def coded_qpsk_channel(n_frames, period, delay, beta, span, esn0_db, msg, rng):
    """tsync_ref.qpsk_channel with the symbols of K = 7 rate-1/2 coded bits: I = 1 - 2 c_0, Q = 1 - 2 c_1"""
    c = R.encode(msg, 7, (0o133, 0o171)).astype(np.float64)
    a = ((1 - 2 * c[:, 0]) + 1j * (1 - 2 * c[:, 1])) / np.sqrt(2)
    n_sym = len(a)
    m = np.arange(n_frames, dtype=np.float64)
    x = np.zeros(n_frames, np.complex128)
    j0 = np.floor((m - delay) / period).astype(np.int64)
    for o in range(-span // 2 - 1, span // 2 + 2):
        j = j0 + o
        ok = (j >= 0) & (j < n_sym)
        x += np.where(ok, a[np.clip(j, 0, n_sym - 1)] * TR.rrc((m - delay - j * period) / period, beta), 0)
    sigma2 = period / 10 ** (esn0_db / 10)
    x += np.sqrt(sigma2 / 2) * (rng.standard_normal(n_frames) + 1j * rng.standard_normal(n_frames))
    return x.astype(np.complex64), a


def quarter_turns(z, r):
    """z i^r exactly, on the host (complex64) or the device (a torch complex64 tensor)"""
    if isinstance(z, np.ndarray):
        re, im = z.real.copy(), z.imag.copy()
        for _ in range(r % 4):
            re, im = -im, re
        return (re + 1j * im).astype(np.complex64)
    import torch
    v = torch.view_as_real(z)
    re, im = v[..., 0], v[..., 1]
    for _ in range(r % 4):
        re, im = -im, re
    return torch.view_as_complex(torch.stack([re, im], -1).contiguous())


def test_ddc_to_tsync_to_eq_to_csync_to_vit_chain(sdr):
    """four RRC QPSK channels carrying K = 7 rate-1/2 coded random bits (I = c_0, Q = c_1), each with the echo pair and
    residual carriers of test_ddc_to_tsync_to_eq_to_csync_chain, in one u8 IQ capture -> sdr_ddc -> sdr_tsync ->
    sdr_eq (CMA) -> sdr_csync (QPSK) -> sdr_vit (uniform start), device-resident.  csync leaves a quarter-turn
    ambiguity and CMA an arbitrary phase: the rotation by i^r that best matches the known symbols over one window is
    applied exactly on the device, and the bit offset is found by correlating against the message.  Zero bit errors
    after acquisition on every channel, and the device chain equals the host-hop chain bit for bit."""
    torch, dev = _torch()
    n, D, Ld, sps = 1 << 22, 16, 255, 64
    freqs = [0.1, -0.27, 0.3, -0.05]
    resid = [0.0, 1e-3, -2e-3, 0.0]
    rng = np.random.default_rng(43)
    x = np.zeros(n, np.complex128)
    msgs, syms = [], []
    for f in freqs:
        delay = rng.uniform(0, sps)
        msg = rng.integers(0, 2, int((n - delay) / sps) + 8 + 2).astype(np.uint8)
        s, a = coded_qpsk_channel(n, sps, delay, 0.35, 8, 80.0, msg, rng)
        msgs.append(msg)
        syms.append(a)
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
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, KD[4] * RADIUS, 1 / (2 * np.pi))
    loop = (4, kp, ki, 2.0 * RADIUS, 0.02)
    cs = sdr.Csync(loop, n_channels=4, stream=st)
    d_z = torch.empty_like(d_sym)
    d_ph = torch.empty((4, cap), dtype=torch.int64, device=dev)
    cs.process_dev(d_q, got, cap, d_z, cap, d_ph, None)
    z = d_z.cpu().numpy()
    # the quarter turn and symbol offset per channel from the known symbols over one window after acquisition
    skip, win = 20000, 2000
    rot, off = [], []
    for k in range(4):
        seg = z[k, skip:skip + win]
        best = None
        for r in range(4):
            zr = quarter_turns(seg, r)
            for d in range(-64, 65):
                ref = syms[k][skip + d:skip + d + win]
                score = (np.sign(zr.real) == np.sign(ref.real)).sum() + (np.sign(zr.imag) == np.sign(ref.imag)).sum()
                if best is None or score > best[0]:
                    best = (score, r, d)
        assert best[0] == 2 * win, (k, best)
        rot.append(best[1])
        off.append(best[2])
    d_r = torch.stack([quarter_turns(d_z[k], rot[k]) for k in range(4)]).contiguous()
    sigma = 64.0
    vit = sdr.Vit(7, (0o133, 0o171), 64, sigma, n_channels=4, zero_start=False, stream=st)
    ocap = cap + 32
    d_b = torch.empty((4, ocap), dtype=torch.uint8, device=dev)
    cnt = vit.process_dev(d_r, got, cap, d_b, ocap)
    bits = d_b.cpu().numpy()
    # the host-hop chain
    hs = sdr.Tsync(taps, P, 4 << 64, tloop, n_channels=4).process(yh)[0]
    hq = sdr.Eq(NTAPS, eadapt, n_channels=4).process(hs)[0]
    hz = sdr.Csync(loop, n_channels=4).process(hq)[0]
    hb = sdr.Vit(7, (0o133, 0o171), 64, sigma, n_channels=4, zero_start=False).process(
        [quarter_turns(hz[k], rot[k]) for k in range(4)])
    for k in range(4):
        g = int(cnt[k])
        assert np.array_equal(bits[k, :g], hb[k])
        # the decoded bit of step i is message bit i + offset
        lo = skip
        dec = bits[k, lo:g]
        ref = msgs[k][lo + off[k]:lo + off[k] + len(dec)]
        errors = int((dec[:len(ref)] != ref).sum())
        print("channel %d: quarter turns %d, offset %d, %d bits checked, %d errors" % (k, rot[k], off[k], len(ref),
                                                                                       errors))
        assert len(ref) > 30000 and errors == 0, (k, errors)

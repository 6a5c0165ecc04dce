"""Frame synchronizer bank (sdr_fsync): payloads, counts and every record field equal the model (fsync_ref) bit for bit
(NaN = NaN) for C in {1, 3, 17, 256, 1024}, Lp in {8, 13, 64, 255, 1024}, W in {0, 1, 4, 32}, V in {0, 1, 3} and
max_miss in {1, 3}, with orders mixed per channel, shared and per-channel words and parameters, F down to
Lp + 2W + 1, and streams with rotations changing between frames, inserted and deleted symbols, missing and false words
and NaN / Inf / zero / overflowing stretches; one-symbol calls, random per-channel splits, calls ending inside a word,
a window or a payload, clones, resets, host against device (one host call spanning several chunks), odd strides and a
retry after OUTPUT_TOO_SMALL give the same bits; at most 2 launches per call; payloads are derotated across a quarter-
turn cycle slip; a deleted symbol is tracked with W = 1 and reacquired with W = 0; the six-stage chain sdr_ddc ->
sdr_tsync -> sdr_eq -> sdr_csync -> sdr_fsync -> sdr_vit with only the sync word known; the C++ mirror; spot channels
at C = 65536."""
import os
import subprocess

import numpy as np
import pytest

import fsync_ref as R
import gen
import tsync_ref as TR
import vit_ref as VR
from test_csync_host import KD
from test_eq_host import EMAX, MU, NTAPS, RADIUS
from test_fsync_host import eventful

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def same_floats(a, b):
    a, b = np.asarray(a, np.float32).ravel(), np.asarray(b, np.float32).ravel()
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all() and (a.view(np.uint32)[~na] == b.view(np.uint32)[~na]).all())


def same_payload(a, b):
    a, b = np.asarray(a, np.complex64), np.asarray(b, np.complex64)
    return a.shape == b.shape and same_floats(a.view(np.float32), b.view(np.float32))


def same_recs(a, b):
    if len(a) != len(b):
        return False
    return all(np.array_equal(a[f], b[f]) for f in ("pos", "out_index", "rot", "kind")) and \
        same_floats(a["corr"], b["corr"]) and same_floats(a["rho"], b["rho"])


def check(got_pay, got_rec, want_pay, want_rec, what=""):
    for k in range(len(want_pay)):
        assert same_recs(got_rec[k], want_rec[k]), (what, k, got_rec[k][:5], want_rec[k][:5])
        assert same_payload(got_pay[k], want_pay[k]), (what, k, len(got_pay[k]), len(want_pay[k]))


def workload(C_, Lp, W, V, mm, seed, n_frames=12, shared_words=False, shared_params=False):
    """(words, params, rows): orders mixed per channel, F from Lp + 2W + 1 up, eventful streams"""
    rng = np.random.default_rng(seed)
    Ms = [(2, 4, 8)[k % 3] for k in range(C_)]
    words = R.word(Lp, rng)[None] if shared_words else np.stack([R.word(Lp, rng, Ms[k]) for k in range(C_)])
    if shared_params:
        params = [(Lp + 2 * W + 1 + int(rng.integers(0, 3)) * 7, 4, 0.6, 0.4, V, mm, W)]
        Ms = [4] * C_
    else:
        params = [(Lp + 2 * W + 1 + (0 if k % 4 == 0 else int(rng.integers(1, 40))), Ms[k], 0.6, 0.4, V, mm, W)
                  for k in range(C_)]
    rows = []
    for k in range(C_):
        prm = params[0 if shared_params else k]
        w = words[0 if shared_words else k]
        rows.append(eventful(w, prm[0], prm[1], n_frames, rng, W, special=k % 2 == 0))
    return words, params, rows


GRID = [(1, 8, 0, 0, 1), (1, 1024, 32, 3, 3), (3, 13, 1, 1, 3), (3, 255, 4, 3, 1), (17, 64, 32, 0, 3),
        (17, 8, 4, 1, 1), (256, 13, 0, 3, 3), (256, 64, 1, 0, 1), (1024, 8, 1, 1, 3), (1024, 64, 4, 3, 1),
        (3, 1024, 0, 1, 1), (17, 255, 1, 0, 3), (256, 8, 32, 1, 3), (1, 64, 4, 3, 3), (1024, 13, 32, 0, 1)]


# every grid point with per-channel words and parameters; shared words or parameters at C = 3 and 256
CASES = [g + ("per_channel",) for g in GRID] + [g + (sh,) for g in GRID if g[0] in (3, 256)
                                                 for sh in ("shared_words", "shared_params")]


@pytest.mark.parametrize("C_,Lp,W,V,mm,sharing", CASES)
def test_fsync_bit_exact_against_the_model(sdr, C_, Lp, W, V, mm, sharing):
    words, params, rows = workload(C_, Lp, W, V, mm, C_ * 1000 + Lp + W * 7 + V * 3 + mm, n_frames=12 if C_ < 256
                                   else 8, shared_words=sharing == "shared_words",
                                   shared_params=sharing == "shared_params")
    want_pay, want_rec = R.model(rows, words, params)
    f = sdr.Fsync(words, params if len(params) > 1 else params[0], n_channels=C_)
    pay, rec = f.process(rows)
    check(pay, rec, want_pay, want_rec)
    b = R.Bank(words, params, C_)
    for k in range(C_):
        b.ch[k].feed(rows[k])
    for k in sorted(set([0, C_ - 1, C_ // 2])):
        assert f.state(k) == b.ch[k].state_tuple(), k
    assert sum(len(r) for r in rec) > C_  # decisions were made


def _dev_call(torch, dev, f, rows, C_, stride=None, rec=True):
    """one process_dev call over rows (a list of C arrays) -> (payload rows, record rows, counts)"""
    n = np.array([len(r) for r in rows])
    stride = stride or max(int(n.max()), 1)
    x = np.zeros((C_, stride), np.complex64)
    for k, r in enumerate(rows):
        x[k, :len(r)] = r
    pc, rc = f.max_output(n)
    cap, rcap = max(int(pc.max()), 1) + 3, max(int(rc.max()), 1) + 1
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_r = torch.empty((C_, rcap, 32), dtype=torch.uint8, device=dev) if rec else None
    got, rgot = f.process_dev(d_x, n, stride, d_y, cap, cap, d_r, rcap, rcap)
    y = d_y.cpu().numpy()
    recs = d_r.cpu().numpy().reshape(C_, rcap * 32).view(R.REC) if rec else None
    return ([y[k, :got[k]].copy() for k in range(C_)],
            [recs[k, :rgot[k]].copy() for k in range(C_)] if rec else None, got, rgot)


def test_fsync_blockings_clone_reset_host_device(sdr):
    torch, dev = _torch()
    C_, Lp, W = 3, 13, 4
    words, params, rows = workload(C_, Lp, W, 1, 3, 77, n_frames=10)
    want_pay, want_rec = R.model(rows, words, params)
    n = [len(r) for r in rows]

    def feed(f, parts_fn, use_dev=False):
        at = [0] * C_
        pays, recs = [[] for _ in range(C_)], [[] for _ in range(C_)]
        i = 0
        while any(a < m for a, m in zip(at, n)):
            take = parts_fn(i, at)
            take = [min(t, m - a) for t, a, m in zip(take, at, n)]
            blk = [rows[k][at[k]:at[k] + take[k]] for k in range(C_)]
            if use_dev:
                p, r, _, _ = _dev_call(torch, dev, f, blk, C_, stride=max(take) + 5)
            else:
                p, r = f.process(blk)
            for k in range(C_):
                pays[k].append(p[k])
                recs[k].append(r[k])
            at = [a + t for a, t in zip(at, take)]
            i += 1
        return ([np.concatenate(p) for p in pays], [np.concatenate(r) for r in recs])

    rng = np.random.default_rng(5)
    # one call, one-symbol calls, random per-channel splits (host and device)
    for parts, use_dev in [(lambda i, at: [max(n)] * C_, False), (lambda i, at: [1] * C_, False),
                           (lambda i, at: [int(rng.integers(0, 60)) for _ in range(C_)], False),
                           (lambda i, at: [int(rng.integers(0, 200)) for _ in range(C_)], True)]:
        f = sdr.Fsync(words, params)
        check(*feed(f, parts, use_dev), want_pay, want_rec)
    # calls ending inside a word, a window and a payload of channel 0
    F0 = params[0][0]
    r0 = want_rec[0]
    cuts = sorted({int(r0["pos"][2]) + Lp // 2, int(r0["pos"][3]) + F0 + Lp + W - 1, int(r0["pos"][4]) + Lp + 5})
    f = sdr.Fsync(words, params)
    got = feed(f, lambda i, at: [cuts[i] - at[0] if i < len(cuts) else max(n)] * C_)
    check(*got, want_pay, want_rec)
    # clone mid-stream, reset
    half = [m // 2 for m in n]
    f = sdr.Fsync(words, params)
    p1, r1 = f.process([rows[k][:half[k]] for k in range(C_)])
    g = f.clone()
    p2, r2 = g.process([rows[k][half[k]:] for k in range(C_)])
    del f
    check([np.concatenate([a, b]) for a, b in zip(p1, p2)], [np.concatenate([a, b]) for a, b in zip(r1, r2)],
          want_pay, want_rec, "clone")
    g.reset()
    assert g.state(0) == (0, 0, 0, 0, 0, 0)
    check(*g.process(rows), want_pay, want_rec, "reset")
    # a retry after OUTPUT_TOO_SMALL leaves the state as it was
    f = sdr.Fsync(words, params)
    f.process([r[:100] for r in rows])
    before = [f.state(k) for k in range(C_)]
    d_x = torch.zeros((C_, 500), dtype=torch.complex64, device=dev)
    d_y = torch.empty((C_, 500), dtype=torch.complex64, device=dev)
    pc, _ = f.max_output(400)
    with pytest.raises(sdr.SdrError) as e:
        f.process_dev(d_x, 400, 500, d_y, int(pc.max()) - 1, 500)
    assert e.value.code == 104 and [f.state(k) for k in range(C_)] == before
    p, r = f.process([r[100:] for r in rows])
    pw, rw = R.model([r[:100] for r in rows], words, params)
    check([np.concatenate([a, b]) for a, b in zip(pw, p)], [np.concatenate([a, b]) for a, b in zip(rw, r)],
          want_pay, want_rec, "retry")


def test_fsync_host_call_spans_chunks(sdr):
    """C = 1024: the host path moves 4096 symbols per channel per round, so 10000 symbols take three rounds"""
    torch, dev = _torch()
    words, params, rows = workload(1024, 16, 2, 1, 2, 91, n_frames=10)
    rows = [np.resize(r, 10000).astype(np.complex64) for r in rows]
    want_pay, want_rec = R.model(rows, words, params)
    check(*sdr.Fsync(words, params).process(rows), want_pay, want_rec, "host")
    p, r, _, _ = _dev_call(torch, dev, sdr.Fsync(words, params), rows, 1024, stride=10001)
    check(p, r, want_pay, want_rec, "device")
    # without records
    f = sdr.Fsync(words, params)
    p, r = f.process(rows, records=False)
    assert r is None and all(same_payload(a, b) for a, b in zip(p, want_pay))


@pytest.mark.parametrize("C_", [1, 1024])
def test_fsync_launch_count(sdr, C_):
    torch, dev = _torch()
    words, params, rows = workload(C_, 32, 2, 1, 2, 5 + C_, n_frames=6)
    f = sdr.Fsync(words, params)
    for part in (slice(0, 150), slice(150, None)):
        before = sdr.kernel_launch_count()
        _dev_call(torch, dev, f, [r[part] for r in rows], C_)
        assert 1 <= sdr.kernel_launch_count() - before <= 2


def test_fsync_cycle_slip_is_derotated(sdr):
    """a quarter-turn slip from frame 7 on: every frame after lock is emitted with its own rotation and the payloads
    equal the transmitted symbols on both sides of the slip"""
    rng = np.random.default_rng(11)
    Lp, F = 64, 64 + 512
    w = R.word(Lp, rng)
    rots = [1] * 7 + [2] * 13
    x, pays = R.framed(w, F, 20, 4, rng, rots, esn0_db=20.0, start=100)
    f = sdr.Fsync(w, (F, 4, 0.5, 0.3, 1, 2, 1))
    pay, rec = f.process(x)
    r = rec[0][rec[0]["out_index"] != R.NO_OUT]
    first = (int(r["pos"][0]) - 100) // F
    assert first <= 2
    assert list(r["rot"]) == rots[first:first + len(r)]
    for j, o in zip(range(first, first + len(r)), r["out_index"]):
        got = pay[0][int(o):int(o) + F - Lp]
        if len(got) == F - Lp:
            assert (np.sign(got.real) == np.sign(pays[j].real)).all() and (np.sign(got.imag) == np.sign(pays[j].imag)).all()
    want = R.model([x], w, (F, 4, 0.5, 0.3, 1, 2, 1))
    check(pay, rec, *want)


def test_fsync_deleted_symbol(sdr):
    """one symbol deleted inside frame 8's payload: with W = 1 the lock holds and LOCK_PASS comes at e - 1; with W = 0
    the lock is lost and reacquired within V + 2 frames"""
    rng = np.random.default_rng(12)
    Lp, F, V = 32, 32 + 400, 1
    w = R.word(Lp, rng)
    x, _ = R.framed(w, F, 20, 4, rng, 0, esn0_db=20.0)
    cut = 8 * F + 200
    x = np.delete(x, cut)
    for W in (1, 0):
        prm = (F, 4, 0.5, 0.3, V, 3 if W else 1, W)
        pay, rec = sdr.Fsync(w, prm).process(x)
        check(pay, rec, *R.model([x], w, prm))
        r = rec[0]
        if W == 1:
            at = r[r["pos"] == 9 * F - 1]
            assert len(at) == 1 and at["kind"][0] == R.LOCK_PASS
            assert not (r["kind"] == R.LOCK_LOST).any()
        else:
            lost = np.nonzero(r["kind"] == R.LOCK_LOST)[0]
            assert len(lost) == 1
            back = r[lost[0] + 1:]
            relock = back[back["out_index"] != R.NO_OUT][0]
            assert (int(relock["pos"]) + 1) % F == 0 and int(relock["pos"]) - int(r["pos"][lost[0]]) <= (V + 2) * F


def test_fsync_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "fsync_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "FSYNC MIRROR OK" in r.stdout, r.stdout + r.stderr


def test_fsync_scale_65536(sdr):
    """C = 65536 shifted copies of one framed stream with per-channel rotations and orders; spot channels match the
    model"""
    torch, dev = _torch()
    C_, Lp, F, n = 65536, 32, 200, 1200
    rng = np.random.default_rng(13)
    w = R.word(Lp, rng)
    base, _ = R.framed(w, F, 9, 4, rng, 0, esn0_db=15.0)
    params = [(F + (k % 5), (2, 4, 8)[k % 3], 0.5, 0.3, k % 3, 1 + k % 3, k % 4) for k in range(C_)]
    shift = (np.arange(C_) * 37) % F
    idx = (np.arange(n)[None, :] + shift[:, None]) % len(base)
    x = base[idx] * np.exp(2j * np.pi * (np.arange(C_) % 4) / 4)[:, None].astype(np.complex64)
    x = x.astype(np.complex64)
    f = sdr.Fsync(w, params)
    pay, rec, got, rgot = _dev_call(torch, dev, f, list(x), C_, stride=n)
    assert rgot.sum() > C_
    for k in [0, 1, 2, 3, 4, 777, 4096, 30001, 65534, 65535]:
        wp, wr = R.model([x[k]], w, params[k])
        check([pay[k]], [rec[k]], wp, wr, k)


# ---- the six-stage chain --------------------------------------------------------------------------------------------

def framed_coded_channel(n_frames_sym, period, delay, beta, span, esn0_db, a, rng):
    """tsync_ref.qpsk_channel's RRC pulse train of the symbols a"""
    n_sym = len(a)
    m = np.arange(n_frames_sym, dtype=np.float64)
    x = np.zeros(n_frames_sym, np.complex128)
    j0 = np.floor((m - delay) / period).astype(np.int64)
    for o in range(-span // 2 - 1, span // 2 + 2):
        j = j0 + o
        ok = (j >= 0) & (j < n_sym)
        x += np.where(ok, a[np.clip(j, 0, n_sym - 1)] * TR.rrc((m - delay - j * period) / period, beta), 0)
    sigma2 = period / 10 ** (esn0_db / 10)
    x += np.sqrt(sigma2 / 2) * (rng.standard_normal(n_frames_sym) + 1j * rng.standard_normal(n_frames_sym))
    return x.astype(np.complex64)


def test_ddc_to_tsync_to_eq_to_csync_to_fsync_to_vit_chain(sdr):
    """four RRC QPSK channels, each a stream of frames of a 64-symbol QPSK word and 1024 symbols of one continuous
    K = 7 rate-1/2 coded message (I = c_0, Q = c_1), with the echo pair and residual carriers of the existing chain, in
    one u8 IQ capture -> sdr_ddc -> sdr_tsync -> sdr_eq (CMA) -> sdr_csync (QPSK) -> sdr_fsync -> sdr_vit, device-
    resident.  Only the word is known: fsync finds the frames and resolves the quarter turn.  Zero bit errors after
    lock on every channel (the test's only freedom is which frame of the message the first payload is), and the device
    chain equals the host-hop chain bit for bit."""
    torch, dev = _torch()
    n, D, Ld, sps = 1 << 22, 16, 255, 64
    Lp, PAY = 64, 1024
    F = Lp + PAY
    freqs = [0.1, -0.27, 0.3, -0.05]
    resid = [0.0, 1e-3, -2e-3, 0.0]
    rng = np.random.default_rng(47)
    word = R.word(Lp, rng)
    x = np.zeros(n, np.complex128)
    msgs = []
    n_frames = n // sps // F + 2
    for f in freqs:
        delay = rng.uniform(0, sps)
        msg = rng.integers(0, 2, n_frames * PAY).astype(np.uint8)
        c = VR.encode(msg, 7, (0o133, 0o171)).astype(np.float64)
        data = ((1 - 2 * c[:, 0]) + 1j * (1 - 2 * c[:, 1])) / np.sqrt(2)
        a = np.concatenate([np.concatenate([word, data[j * PAY:(j + 1) * PAY]]) for j in range(n_frames)])
        msgs.append(msg)
        s = framed_coded_channel(n, sps, delay, 0.35, 8, 80.0, a, rng).astype(np.complex128)
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
    cs.process_dev(d_q, got, cap, d_z, cap)
    fprm = (F, 4, 0.5, 0.3, 1, 3, 2)
    fs = sdr.Fsync(word, fprm, n_channels=4, stream=st)
    pcap, rcap = (int(v.max()) for v in fs.max_output(got))
    d_p = torch.empty((4, pcap), dtype=torch.complex64, device=dev)
    d_rec = torch.empty((4, rcap, 32), dtype=torch.uint8, device=dev)
    npay, nrec = fs.process_dev(d_z, got, cap, d_p, pcap, pcap, d_rec, rcap, rcap)
    recs = d_rec.cpu().numpy().reshape(4, rcap * 32).view(R.REC)
    sigma = 64.0
    vit = sdr.Vit(7, (0o133, 0o171), 64, sigma, n_channels=4, zero_start=False, stream=st)
    ocap = (pcap + 35) // 4 * 4  # device rows are 4-byte aligned
    d_b = torch.empty((4, ocap), dtype=torch.uint8, device=dev)
    cnt = vit.process_dev(d_p, npay, pcap, d_b, ocap)
    bits = d_b.cpu().numpy()
    # the host-hop chain
    hs = sdr.Tsync(taps, P, 4 << 64, tloop, n_channels=4).process(yh)[0]
    hq = sdr.Eq(NTAPS, eadapt, n_channels=4).process(hs)[0]
    hz = sdr.Csync(loop, n_channels=4).process(hq)[0]
    hp, hr = sdr.Fsync(word, fprm, n_channels=4).process(hz)
    hb = sdr.Vit(7, (0o133, 0o171), 64, sigma, n_channels=4, zero_start=False).process(hp)
    for k in range(4):
        r = recs[k, :nrec[k]]
        assert same_recs(r, hr[k]) and same_payload(d_p[k, :npay[k]].cpu().numpy(), hp[k])
        g = int(cnt[k])
        assert np.array_equal(bits[k, :g], hb[k])
        # payload i after the first emitted frame is coded symbol j0 PAY + i; skip 24 frames of acquisition
        skip = 24 * PAY
        dec = bits[k, skip:g]
        best = None
        for j0 in range(n_frames):
            ref = msgs[k][j0 * PAY + skip:j0 * PAY + skip + len(dec)]
            if len(ref) < len(dec) // 2:
                break
            e = int((dec[:len(ref)] != ref).sum())
            if best is None or e < best[0]:
                best = (e, j0, len(ref))
        kinds = np.bincount(r["kind"], minlength=7)[1:]
        print("channel %d: first frame %d, %d bits checked, %d errors; records HIT/VP/VF/LP/LM/LL %s" % (
            k, best[1], best[2], best[0], list(kinds)))
        assert best[2] > 25000 and best[0] == 0, (k, best)

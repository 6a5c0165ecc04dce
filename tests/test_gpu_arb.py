"""Arbitrary-ratio resampler bank (sdr_arb): every output against the f64 definition at exact positions; bit-exact
agreement with sdr_rrb on its grid; bit-exact known answers; no drift over 2^26 frames (spot outputs and a tone's phase);
blockings, clones, resets, retries, strides, host against device and output-anchored shards; set_steps against the
piecewise definition; NaN bounds; the launch count; device-resident chains from sdr_ddc and sdr_pfb; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import arb_ref as A
import gen

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ONE = A.ONE

PPM_UP = A.step_of(1 + 37e-6, 1.0)
STEPS = [PPM_UP, A.step_of(1 - 37e-6, 1.0), A.step_of(48000.0, 44100.0), A.step_of(44100.0, 48000.0),
         A.step_of(6.25 * (1 + 37e-6), 1.0), A.step_of(1.0, 4.41), ONE]


def _bar(z64):
    return 1e-5 * max(np.abs(z64).max(), 1e-30)


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
    """0, random 64.64 values below 3 frames and random whole parts below 40"""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(C_):
        f = int(rng.integers(0, 1 << 64, dtype=np.uint64))
        out.append([0, f % (3 * ONE), (int(rng.integers(0, 40)) << 64) | (f & A.MASK)][k % 3])
    return out


def _z64(h, P, row, taus, chunk=4096):
    """the f64 definition (computed form, exact weights) at exact positions; row: numpy or a torch row on the device"""
    L = h.size
    out = []
    for s in range(0, len(taus), chunk):
        part = taus[s:s + chunk]
        at = max(0, (part[0] >> 64) - -(-L // P) - 1)
        end = (part[-1] >> 64) + 1
        y = row[at:end]
        y = y.cpu().numpy() if hasattr(y, "cpu") else y
        out.append(A.computed_f64(h, P, np.asarray(y, np.complex128), part, at=at))
    return np.concatenate(out) if out else np.zeros(0, np.complex128)


def _check(got, h, P, y, firsts, steps):
    for k in range(len(got)):
        hk = A.taps_of(h, k).astype(np.float64)
        n = A.released(y[k].size if isinstance(y, list) else y.shape[1], firsts[k], steps[k])
        assert got[k].shape == (n,), k
        if n == 0:
            continue
        z64 = _z64(hk, P, y[k], [firsts[k] + r * steps[k] for r in range(n)])
        assert np.abs(got[k] - z64).max() <= _bar(z64), k


@pytest.mark.parametrize("C_,P,L,shared", [
    (1, 1, 1, True), (1, 32, 8195, True), (1, 4096, 65537, True), (3, 2, 7, False), (3, 256, 4096, False),
    (3, 1, 255, True), (17, 32, 255, False), (17, 4096, 8195, True), (256, 256, 255, True), (256, 1, 7, False),
    (1024, 32, 255, True), (1024, 2, 7, False)])
def test_arb_against_f64(sdr, C_, P, L, shared):
    steps = [STEPS[(k + L) % len(STEPS)] for k in range(C_)]
    firsts = _firsts(C_, C_ + L)
    h = _taps(C_, L, P, shared, C_ + P)
    nf = 3000 if C_ <= 17 else 300
    y = _rows(C_, nf, C_ + L + P)
    got = sdr.Arb(h, P, steps, firsts).process(y)
    assert len(got) == C_
    _check(got, h, P, y, firsts, steps)


def test_arb_range_end_steps(sdr):
    """sigma = 2^-16 (65536 outputs per frame) and 2^24, per-channel frame counts in one call"""
    torch, dev = _torch()
    P, L = 2, 7
    h = _taps(1, L, P, True, 1)
    steps, firsts = [1 << 48, 1 << 88], [0, ONE // 3]
    n = [12, (1 << 25) + 3]
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(3)
    d_y = torch.randn((2, n[1]), dtype=torch.complex64, device=dev, generator=g)
    b = sdr.Arb(h, P, steps, firsts, stream=st)
    cnt = b.output_count(n)
    assert list(cnt) == [A.released(n[0], firsts[0], steps[0]), 3] and cnt[0] == 12 * 65536
    cap = int(cnt.max())
    d_z = torch.empty((2, cap), dtype=torch.complex64, device=dev)
    assert list(b.process_dev(d_y, n, n[1], d_z, cap, cap)) == list(cnt)
    torch.cuda.synchronize()
    for k in range(2):
        z64 = _z64(h.astype(np.float64), P, d_y[k], [firsts[k] + r * steps[k] for r in range(int(cnt[k]))],
                   chunk=4096 if k == 0 else 1)
        got = d_z[k, :int(cnt[k])].cpu().numpy()
        assert np.abs(got - z64).max() <= _bar(z64), k
    del d_y, d_z


def test_arb_counts_at_whole_parts_of_2_40(sdr):
    """first positions with whole parts of 2^40: the exact counts at frame totals near 2^40"""
    big = (1 << 40 << 64) | 0x5555555555555555
    b = sdr.Arb(_taps(1, 33, 8, True), 8, [PPM_UP, A.step_of(1.0, 4.41), 1 << 88], [big, big + 7, big], n_channels=3)
    for n in (1 << 40, (1 << 40) + 1, (1 << 40) + 12345):
        assert list(b.output_count(n)) == [A.released(n, f, s) for f, s in
                                           zip([big, big + 7, big], [PPM_UP, A.step_of(1.0, 4.41), 1 << 88])]
    assert list(b.output_count(1 << 40)) == [0, 0, 0]


@pytest.mark.parametrize("I", [2, 8, 32])
def test_arb_equals_rrb_bits(sdr, I):
    """P = I, sigma = D / I, tau(0) = ((r0+1) D - I) / I: sdr_rrb's outputs from r0 on, bit for bit; its first r0 are 0"""
    Ds = [1, 3, 25, 147]
    L = 255
    h = _taps(1, L, I, True, I)
    y = _rows(len(Ds), 4000, I)
    zr = sdr.Rrb(h, I, Ds).process(y)
    firsts = [A.rrb_first(I, D)[1] for D in Ds]
    za = sdr.Arb(h, I, [D * ONE // I for D in Ds], firsts).process(y)
    for k, D in enumerate(Ds):
        r0 = A.rrb_first(I, D)[0]
        assert (zr[k][:r0] == 0).all()
        common = min(za[k].size, zr[k].size - r0)
        assert common > 0 and za[k].size >= zr[k].size - r0
        assert np.array_equal(_bits(za[k][:common]), _bits(zr[k][r0:r0 + common])), D


@pytest.mark.parametrize("step,first", [(1, 0), (2, 3), (3, 10), (7, 1)])
def test_arb_known_answers_bit_exact(sdr, step, first):
    """P = 1, L = 1, h = [a], integer sigma and tau(0): z[r] = f32(a y[tau(0) + r sigma])"""
    a = np.float32(-0.7734375)
    y = _rows(3, 2000, step)
    z = sdr.Arb(np.array([a], np.float32), 1, step * ONE, first * ONE, n_channels=3).process(y)
    r = np.arange(A.released(2000, first * ONE, step * ONE))
    for k in range(3):
        yk = y[k][first + r * step]
        want = np.empty(r.size, np.complex64)
        want.real = a * yk.real
        want.imag = a * yk.imag
        assert np.array_equal(_bits(z[k]), _bits(want))


def _tone_gain(h, P, nu, fracs):
    """G(phi) = sum_i H(i + phi) exp(-2 pi j nu (i + phi)): the steady-state response to exp(2 pi j nu m) at fraction
    phi, so that z[r] = exp(2 pi j nu tau(r)) G(frac(tau(r)))"""
    L = h.size
    hx = np.append(h, 0.0)
    T = -(-L // P)
    out = []
    for phi in fracs:
        t = np.arange(T) + phi
        tp = t * P
        j = np.floor(tp).astype(np.int64)
        a = tp - j
        ok = j < L
        jj = np.minimum(j, L - 1)
        Ht = np.where(ok, (1 - a) * hx[jj] + a * hx[jj + 1], 0)
        out.append((Ht * np.exp(-2j * np.pi * nu * t)).sum())
    return np.array(out)


def test_arb_no_drift_over_2_26_frames(sdr):
    """sigma = 1 + 37 ppm over 2^26 frames in one call: spot outputs at the end (about 2500 frames of accumulated
    offset) match f64 at exact positions, and a tone's output phase tracks 2 pi nu tau(r) within the prototype's
    interpolation error"""
    torch, dev = _torch()
    P, L = 256, 4096
    h = _taps(1, L, P, True, 5)
    n = 1 << 26
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(11)
    d_y = torch.empty((2, n), dtype=torch.complex64, device=dev)
    d_y[0] = torch.randn(n, dtype=torch.complex64, device=dev, generator=g)
    tone = torch.from_numpy(np.exp(2j * np.pi * np.arange(64) / 64).astype(np.complex64)).to(dev)  # nu = 1/64
    d_y[1] = tone[torch.arange(n, device=dev) % 64]
    b = sdr.Arb(h, P, PPM_UP, n_channels=2, stream=st)
    cnt = A.released(n, 0, PPM_UP)
    assert n - cnt > 2400
    d_z = torch.empty((2, cnt), dtype=torch.complex64, device=dev)
    assert list(b.process_dev(d_y, n, n, d_z, cnt, cnt)) == [cnt, cnt]
    torch.cuda.synchronize()
    hh = h.astype(np.float64)
    for r0 in (0, cnt // 2 + 333, cnt - 4096):
        taus = [r * PPM_UP for r in range(r0, r0 + 4096)]
        z64 = _z64(hh, P, d_y[0], taus)
        got = d_z[0, r0:r0 + 4096].cpu().numpy()
        assert np.abs(got - z64).max() <= _bar(z64), r0
    # the tone: z[r] exp(-2 pi j tau(r) / 64) = G(frac tau(r)); its phase stays within G's spread over fractions
    nu = 1.0 / 64
    G = _tone_gain(hh, P, nu, np.arange(1024) / 1024.0)
    ref = np.angle(G.mean())
    spread = np.abs(np.angle(G * np.exp(-1j * ref))).max()
    for r0 in (L // P + 8, cnt // 2, cnt - 4096):
        r = np.arange(r0, r0 + 4096)
        taus = [int(x) * PPM_UP for x in r]
        ph = np.array([2 * np.pi * ((t % (64 * ONE)) / (64 * ONE)) for t in taus])
        z = d_z[1, r0:r0 + 4096].cpu().numpy().astype(np.complex128) * np.exp(-1j * ph)
        err = np.abs(np.angle(z * np.exp(-1j * ref)))
        assert err.max() <= 1.1 * spread + 1e-5, (r0, err.max(), spread)
    del d_y, d_z


def test_arb_blockings_clone_reset_retry_strides(sdr):
    C_, P, L = 5, 32, 255
    steps = [PPM_UP, A.step_of(48000.0, 44100.0), A.step_of(1.0, 4.41), A.step_of(6.25, 1.0), ONE]
    firsts = _firsts(C_, 7)
    h = _taps(C_, L, P, False, 9)
    nf = 1500
    y = _rows(C_, nf, 10)
    one = sdr.Arb(h, P, steps, firsts).process(y)
    # 1-frame calls
    p = sdr.Arb(h, P, steps, firsts)
    parts = [p.process(y[:, m:m + 1]) for m in range(300)]
    rest = p.process(y[:, 300:])
    for k in range(C_):
        assert np.array_equal(_bits(np.concatenate([q[k] for q in parts] + [rest[k]])), _bits(one[k]))
    # random splits, different per channel, with a clone mid-stream
    rng = np.random.default_rng(L)
    p = sdr.Arb(h, P, steps, firsts)
    pos = np.zeros(C_, np.int64)
    outs = [[] for _ in range(C_)]
    clone = None
    while (pos < nf).any():
        take = np.minimum(nf - pos, rng.integers(0, 90, C_))
        got = p.process([y[k, pos[k]:pos[k] + take[k]] for k in range(C_)])
        for k in range(C_):
            outs[k].append(got[k])
        pos += take
        if clone is None and pos.min() > nf // 2:
            clone, at, made = p.clone(), pos.copy(), [sum(o.size for o in outs[k]) for k in range(C_)]
    for k in range(C_):
        assert np.array_equal(_bits(np.concatenate(outs[k])), _bits(one[k]))
    cz = clone.process([y[k, at[k]:] for k in range(C_)])
    for k in range(C_):
        assert np.array_equal(_bits(cz[k]), _bits(one[k][made[k]:]))
    p.reset()
    again = p.process(y)
    for k in range(C_):
        assert np.array_equal(_bits(again[k]), _bits(one[k]))
    # a too-small out_cap is refused before any state changes, host and device; the retry gives the same bits
    torch, dev = _torch()
    p = sdr.Arb(h, P, steps, firsts)
    first = p.process(y[:, :7])
    restm = np.ascontiguousarray(y[:, 7:])
    n = np.full(C_, restm.shape[1], np.uintp)
    cap = int(p.output_count(restm.shape[1]).max())
    out = np.empty((C_, cap), np.complex64)
    got = np.zeros(C_, np.uintp)
    rc = sdr.lib().sdr_arb_process(p.h, restm.ctypes.data, n.ctypes.data, restm.shape[1], out.ctypes.data, cap - 1,
                                   cap, got.ctypes.data)
    assert rc == 104 and not got.any()
    d_in = torch.from_numpy(restm).to(dev)
    d_out = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_arb_process_dev(p.h, d_in.data_ptr(), n.ctypes.data, restm.shape[1], d_out.data_ptr(), cap - 1,
                                       cap, got.ctypes.data)
    assert rc == 104 and not got.any()
    second = p.process(restm)
    for k in range(C_):
        assert np.array_equal(_bits(np.concatenate([first[k], second[k]])), _bits(one[k]))
    # odd device strides give the host bits, and nothing past the counts is written
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = y
    d_y = torch.from_numpy(pad).to(dev)
    cap = max(o.size for o in one)
    d_out = torch.full((C_, cap + 3), float("nan"), dtype=torch.complex64, device=dev)
    got = sdr.Arb(h, P, steps, firsts, stream=st).process_dev(d_y, nf, nf + 5, d_out, cap, cap + 3)
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    for k in range(C_):
        assert got[k] == one[k].size
        assert np.array_equal(_bits(out[k, :got[k]]), _bits(one[k])) and np.isnan(out[k, got[k]:]).all()
    # misaligned device pointers are refused
    n = np.full(C_, nf, np.uintp)
    got = np.zeros(C_, np.uintp)
    fresh = sdr.Arb(h, P, steps, firsts)
    rc = sdr.lib().sdr_arb_process_dev(fresh.h, d_y.data_ptr() + 4, n.ctypes.data, nf + 5, d_out.data_ptr(), cap + 3,
                                       cap + 3, got.ctypes.data)
    assert rc == 105 and not got.any()


def test_arb_host_call_larger_than_the_chunk(sdr):
    """one host call of more frames than the host path moves per round gives process_dev's bits"""
    torch, dev = _torch()
    C_, P, L = 2, 64, 1024
    steps = [A.step_of(48000.0, 44100.0), A.step_of(1.0, 4.41)]
    h = _taps(1, L, P, True, 12)
    nf = (1 << 21) + 777  # the host path moves 2^21 frames per channel per round at C = 2
    y = _rows(C_, nf, 13)
    host = sdr.Arb(h, P, steps).process(y)
    st = torch.cuda.current_stream(dev)
    b = sdr.Arb(h, P, steps, stream=st)
    cnt = b.output_count(nf)
    cap = int(cnt.max())
    d_y = torch.from_numpy(y).to(dev)
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    assert list(b.process_dev(d_y, nf, nf, d_z, cap, cap)) == list(cnt)
    torch.cuda.synchronize()
    z = d_z.cpu().numpy()
    for k in range(C_):
        assert host[k].size == cnt[k]
        assert np.array_equal(_bits(host[k]), _bits(z[k, :cnt[k]]))
    del d_y, d_z


def test_arb_output_anchored_shards(sdr):
    C_, P, L = 4, 32, 1023
    steps = [PPM_UP, A.step_of(48000.0, 44100.0), A.step_of(1.0, 4.41), A.step_of(147.0, 160.0)]
    firsts = _firsts(C_, 14)
    h = _taps(C_, L, P, False, 15)
    nf = 8000
    y = _rows(C_, nf, 16)
    one = sdr.Arb(h, P, steps, firsts).process(y)
    T = -(-L // P)
    for world in (2, 3, 5):
        parts = [[] for _ in range(C_)]
        for s in range(world):
            R0 = [one[k].size * s // world for k in range(C_)]
            R1 = [one[k].size * (s + 1) // world for k in range(C_)]
            tau0 = [firsts[k] + R0[k] * steps[k] for k in range(C_)]
            f = max(0, min((t >> 64) - T + 1 for t in tau0))
            ends = [((firsts[k] + (R1[k] - 1) * steps[k]) >> 64) + 1 for k in range(C_)]
            z = sdr.Arb(h, P, steps, [t - f * ONE for t in tau0]).process([y[k, f:max(ends[k], f)] for k in range(C_)])
            for k in range(C_):
                assert z[k].size >= R1[k] - R0[k]
                parts[k].append(z[k][:R1[k] - R0[k]])
        for k in range(C_):
            assert np.array_equal(_bits(np.concatenate(parts[k])), _bits(one[k])), (world, k)


def test_arb_set_steps(sdr):
    """a change applies from the next unreleased output on: against the piecewise definition, and two blockings that put
    the change at the same output index give the same bits"""
    C_, P, L = 3, 32, 255
    steps = [PPM_UP, A.step_of(48000.0, 44100.0), A.step_of(1.0, 4.41)]
    new = [A.step_of(1 - 37e-6, 1.0), A.step_of(44100.0, 48000.0), A.step_of(4.41, 1.0)]
    firsts = _firsts(C_, 17)
    h = _taps(1, L, P, True, 18)
    nf = 3000
    y = _rows(C_, nf, 19)
    # channel 1 (sigma > 1): a frame count whose last frame releases nothing, so fewer frames reach the same index
    a = [1000, next(m for m in range(1333, 1400) if A.released(m, firsts[1], steps[1]) ==
                    A.released(m - 1, firsts[1], steps[1])), 777]
    tbs = [A.Timebase(firsts[k], steps[k]) for k in range(C_)]
    for k in range(C_):
        tbs[k].set_step(a[k], new[k])
    p = sdr.Arb(h, P, steps, firsts)
    z1 = p.process([y[k, :a[k]] for k in range(C_)])
    p.set_steps(new)
    z2 = p.process([y[k, a[k]:] for k in range(C_)])
    full = [np.concatenate([z1[k], z2[k]]) for k in range(C_)]
    for k in range(C_):
        n = tbs[k].released(nf)
        assert full[k].size == n
        z64 = _z64(h.astype(np.float64), P, y[k], [tbs[k].tau(r) for r in range(n)])
        assert np.abs(full[k] - z64).max() <= _bar(z64), k
    # the same change index after fewer frames (just enough to release the same outputs), in different calls
    b = [min(m for m in range(a[k] + 1) if A.released(m, firsts[k], steps[k]) == A.released(a[k], firsts[k], steps[k]))
         for k in range(C_)]
    assert b != a
    q = sdr.Arb(h, P, steps, firsts)
    w = [[] for _ in range(C_)]
    for lo, hi in ((0, 0.5), (0.5, 1.0)):
        got = q.process([y[k, int(b[k] * lo):int(b[k] * hi)] for k in range(C_)])
        for k in range(C_):
            w[k].append(got[k])
    q.set_steps(new)
    got = q.process([y[k, b[k]:] for k in range(C_)])
    for k in range(C_):
        w[k].append(got[k])
    for k in range(C_):
        assert np.array_equal(_bits(np.concatenate(w[k])), _bits(full[k])), k
    # reset restores the creation steps, a clone copies the current ones
    p.reset()
    again = p.process(y)
    ref = sdr.Arb(h, P, steps, firsts).process(y)
    for k in range(C_):
        assert np.array_equal(_bits(again[k]), _bits(ref[k]))


@pytest.mark.parametrize("P,L", [(1, 64), (32, 255), (256, 4096)])
def test_arb_nan_poisons_exactly_its_outputs(sdr, P, L):
    C_ = 2
    steps = [A.step_of(48000.0, 44100.0), A.step_of(1.0, 4.41)]
    firsts = [0, ONE // 7]
    h = _taps(C_, L, P, False, 20)
    h[1][L // 2] = 0.0
    T = -(-L // P)
    nf = 8 * T + 400
    y = _rows(C_, nf, 21)
    m = nf // 2
    bad = y.copy()
    bad[1, m] = np.complex64(complex(np.nan, 0.0))
    z = sdr.Arb(h, P, steps, firsts).process(bad)
    ref = sdr.Arb(h, P, steps, firsts).process(y)
    taus = [firsts[1] + r * steps[1] for r in range(z[1].size)]
    hit = np.array([(t >> 64) - A.terms(P, L, t) + 1 <= m <= (t >> 64) for t in taus])
    assert hit.any() and not hit.all()
    assert np.isnan(z[1][hit].real).all()
    assert np.array_equal(_bits(z[1][~hit]), _bits(ref[1][~hit]))
    assert np.array_equal(_bits(z[0]), _bits(ref[0]))


@pytest.mark.parametrize("C_", [1, 1024])
def test_arb_launch_count(sdr, C_):
    torch, dev = _torch()
    steps = [STEPS[k % len(STEPS)] for k in range(C_)]
    b = sdr.Arb(_taps(1, 255, 32, True, 22), 32, steps)
    n = 2000
    d_y = torch.randn((C_, n), dtype=torch.complex64, device=dev)
    cap = int(b.output_count(n).max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    before = sdr.kernel_launch_count()
    b.process_dev(d_y, n, n, d_z, cap, cap)
    assert sdr.kernel_launch_count() - before <= 2
    torch.cuda.synchronize()


def test_ddc_to_arb_chain(sdr):
    """sdr_ddc (u8, tensor path, D = 8) at 2.4 MS/s -> sdr_arb at 6.25 (1 + 37 ppm): 48 kHz with clock correction,
    device-resident, equals the host-hop chain bit for bit"""
    torch, dev = _torch()
    n, D, Ld = 1 << 22, 8, 255
    freqs = [0.1, -0.27]
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0)
    P, L = 256, 8192
    step = A.step_of(6.25 * (1 + 37e-6), 1.0)
    ha = _taps(1, L, P, True, 23)
    raw = gen.random_u8(2 * n, 24)
    st = torch.cuda.current_stream(dev)
    ddc = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    nf = n // D
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((2, nf), dtype=torch.complex64, device=dev)
    assert ddc.process_dev(d_in, n, d_y, nf, nf) == nf
    assert ddc.last_path == 2
    arb = sdr.Arb(ha, P, step, n_channels=2, stream=st)
    cnt = A.released(nf, 0, step)
    d_z = torch.empty((2, cnt), dtype=torch.complex64, device=dev)
    assert list(arb.process_dev(d_y, nf, nf, d_z, cnt, cnt)) == [cnt, cnt]
    torch.cuda.synchronize()
    yh = d_y.cpu().numpy()
    host = sdr.Arb(ha, P, step, n_channels=2).process(yh)
    z = d_z.cpu().numpy()
    for k in range(2):
        assert np.array_equal(_bits(z[k]), _bits(host[k])), k
        r = np.arange(cnt - 2048, cnt)
        z64 = _z64(ha.astype(np.float64), P, yh[k], [int(x) * step for x in r])
        assert np.abs(z[k][r] - z64).max() <= _bar(z64), k


def test_pfb_channel_major_to_arb(sdr):
    """sdr_pfb's channel-major rows at M = 1024 go straight in, each channel with its own step"""
    torch, dev = _torch()
    M, D, Lp = 1024, 512, 8 * 1024
    hp = gen.lowpass_taps(Lp, 0.5 / M, 1.0)
    n = 1 << 21
    x = gen.complex_noise(n, 25)
    st = torch.cuda.current_stream(dev)
    pfb = sdr.Pfb(hp, M, D, "c64", channel_major=True, stream=st)
    nf = pfb.output_count(n)
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.empty((M, nf), dtype=torch.complex64, device=dev)
    assert pfb.process_dev(d_x, n, d_y, nf) == nf
    steps = [STEPS[k % len(STEPS)] for k in range(M)]
    P, L = 32, 255
    h = _taps(1, L, P, True, 26)
    arb = sdr.Arb(h, P, steps, stream=st)
    cnt = arb.output_count(nf)
    cap = int(cnt.max())
    d_z = torch.empty((M, cap), dtype=torch.complex64, device=dev)
    assert list(arb.process_dev(d_y, nf, nf, d_z, cap, cap)) == list(cnt)
    torch.cuda.synchronize()
    yh = d_y.cpu().numpy()
    host = sdr.Arb(h, P, steps).process(yh)
    z = d_z.cpu().numpy()
    for k in range(M):
        assert np.array_equal(_bits(z[k, :cnt[k]]), _bits(host[k])), k
    for k in (0, 1, 5, M - 1):
        z64 = _z64(h.astype(np.float64), P, yh[k], [r * steps[k] for r in range(int(cnt[k]))])
        assert np.abs(host[k] - z64).max() <= _bar(z64), k


def test_arb_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "arb_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ARB MIRROR OK" in r.stdout, r.stdout + r.stderr

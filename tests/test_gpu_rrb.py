"""Rational resampler bank (sdr_rrb): against the f64 computed form and the crate's own composition (zero-stuff,
Fir(h_k), decimate) through the CPU oracle; bit-exact known answers; agreement with sdr_fir (I = 1), sdr_duc (D = 1) and
the reduced ratio; blockings, clones, resets, strides and primed shards; errors, NaN bounds and the launch count;
device-resident chains with sdr_ddc, sdr_fcfb and sdr_duc; spot outputs at 2^26 and the C++ mirror."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import scipy.signal

import ddc_ref
import gen
import oracle_lib as O
import rrb_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bar(z64):
    return 1e-5 * max(np.abs(z64).max(), 1e-30)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _ratios(C_, seed):
    """per-channel (I, D) drawn from the ratios users need, with gcd > 1 and 1/1 among them"""
    pool = [(4, 25), (147, 160), (75, 64), (2, 25), (1, 5), (3, 4), (1, 1), (6, 4), (5, 1), (147, 8000), (12, 18)]
    rng = np.random.default_rng(seed)
    pick = [pool[i % len(pool)] for i in range(C_)] if C_ <= len(pool) else [pool[i] for i in
                                                                               rng.integers(0, len(pool), C_)]
    return [p[0] for p in pick], [p[1] for p in pick]


def _taps(C_, L, Is, shared, seed=0):
    """low-pass taps with DC gain I (cutoff 0.45 / max(I, D)), one row per channel unless shared"""
    rng = np.random.default_rng(seed)
    rows = []
    for k in range(1 if shared else C_):
        t = gen.lowpass_taps(L, 0.2 + 0.05 * rng.random(), 1.0) if L > 1 else np.ones(1)
        rows.append(Is[k] * t / t.sum())
    t = np.asarray(rows, np.float32)
    return t[0] if shared else t


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n)


def _check_channels(got, h, y, Is, Ds, oracle=True):
    for k in range(len(Is)):
        hk = R.taps_of(h, k).astype(np.float64)
        z64 = R.computed_f64(hk, y[k], Is[k], Ds[k])
        assert got[k].shape == z64.shape, k
        if z64.size == 0:
            continue
        assert np.abs(got[k] - z64).max() <= _bar(z64), k
        if oracle:
            zo = R.oracle_f32(R.taps_of(h, k), y[k], Is[k], Ds[k])
            assert np.abs(got[k] - zo).max() <= _bar(z64), k


@pytest.mark.parametrize("C_,L,shared,mixed", [
    (1, 255, True, False), (1, 4095, True, True), (3, 64, False, True), (3, 1, True, True), (17, 511, False, True),
    (17, 1023, True, True), (256, 97, True, False), (256, 255, False, True), (1024, 97, True, False),
    (1024, 33, False, True)])
def test_rrb_against_f64_and_oracle(sdr, C_, L, shared, mixed):
    if mixed:
        Is, Ds = _ratios(C_, C_ + L)
    else:
        Is, Ds = [3] * C_, [4] * C_
    h = _taps(C_, L, Is if not shared else [Is[0]] * C_, shared, C_)
    nf = 3000 if C_ <= 17 else 400
    nf = max(nf, 2 * max(Ds) // min(Is) + 8) if C_ <= 17 else nf
    y = _rows(C_, nf, C_ + L)
    got = sdr.Rrb(h, Is, Ds).process(y)
    assert len(got) == C_
    _check_channels(got, h, y, Is, Ds, oracle=C_ <= 17)


@pytest.mark.parametrize("I,D,L", [(4, 25, 4095), (1, 3, 1000), (2, 1, 2001)])
def test_rrb_long_chains(sdr, I, D, L):
    """ceil(L / I) up to about 1000 taps per output"""
    h = _taps(1, L, [I], True, L)
    y = _rows(1, 6000, L)
    got = sdr.Rrb(h, I, D).process(y)
    _check_channels(got, h, y, [I], [D])


@pytest.mark.parametrize("I,D", [(4, 25), (75, 64), (3, 4), (7, 2), (5, 1), (1, 3)])
def test_rrb_known_answers_bit_exact(sdr, I, D):
    """h = ones(I): z[r] = y[((r+1) D div I) - 1]; L = 1, h = [a]: z[r] = a y[q - 1] when c = 0, else 0"""
    C_ = 3
    y = _rows(C_, 2000, I + D)
    z = sdr.Rrb(np.ones(I, np.float32), I, D, n_channels=C_).process(y)
    r = np.arange(R.released(2000, I, D))
    for k in range(C_):
        want = np.concatenate([[0], y[k]]).astype(np.complex64)[((r + 1) * D) // I]
        assert np.array_equal(_bits(z[k]), _bits(want))
    a = np.float32(-0.7734375)
    z = sdr.Rrb(np.array([a], np.float32), I, D, n_channels=C_).process(y)
    t1 = (r + 1) * D
    q, c = t1 // I, t1 % I
    for k in range(C_):
        yk = np.concatenate([[0], y[k]]).astype(np.complex64)[q]
        want = np.zeros(r.size, np.complex64)
        want.real = np.where(c == 0, a * yk.real, 0)
        want.imag = np.where(c == 0, a * yk.imag, 0)
        assert np.array_equal(z[k], want)


@pytest.mark.parametrize("C_,D,L", [(1, 5, 255), (8, 10, 64), (3, 1, 100)])
def test_rrb_interpolation_1_agrees_with_fir(sdr, C_, D, L):
    h = _taps(1, L, [1], True, 3)
    y = _rows(C_, 20000, 4)
    z = sdr.Rrb(h, 1, D, n_channels=C_).process(y)
    f = sdr.Fir(h, "c64", decimation=D, n_channels=C_).process(y)
    f = f.reshape(C_, -1)
    for k in range(C_):
        z64 = R.computed_f64(h.astype(np.float64), y[k], 1, D)
        n = min(z[k].size, f[k].size)
        assert n >= z64.size - 1
        assert np.abs(z[k][:n] - f[k][:n]).max() <= 2 * _bar(z64)


@pytest.mark.parametrize("I,L", [(8, 255), (10, 1000), (3, 1)])
def test_rrb_decimation_1_equals_duc(sdr, I, L):
    h = _taps(1, L, [I], True, 5)
    y = _rows(1, 3000, 6)
    z = sdr.Rrb(h, I, 1).process(y)[0]
    x = sdr.Duc(h, [0.0], 1.0, I).process(y)
    assert np.array_equal(z, x)


@pytest.mark.parametrize("I,D,g,L", [(4, 25, 3, 301), (147, 160, 2, 3529), (1, 5, 4, 255), (3, 1, 5, 40)])
def test_rrb_reduced_ratio_same_bits(sdr, I, D, g, L):
    h = _taps(1, L, [g * I], True, 7)
    y = _rows(2, 5000, 8)
    a = sdr.Rrb(h, g * I, g * D, n_channels=2).process(y)
    b = sdr.Rrb(np.ascontiguousarray(h[::g]), I, D, n_channels=2).process(y)
    for k in range(2):
        assert a[k].size == R.released(5000, I, D)
        assert np.array_equal(_bits(a[k]), _bits(b[k]))


@pytest.mark.parametrize("L,shared", [(255, False), (33, True), (1, True)])
def test_rrb_blockings_clone_reset_retry(sdr, L, shared):
    C_ = 5
    Is, Ds = [4, 147, 75, 1, 7], [25, 160, 64, 5, 7]
    h = _taps(C_, L, Is, shared, 9)
    nf = 1500
    y = _rows(C_, nf, 10)
    one = sdr.Rrb(h, Is, Ds).process(y)
    # 1-frame calls
    p = sdr.Rrb(h, Is, Ds)
    parts = [p.process(y[:, m:m + 1]) for m in range(300)]
    rest = p.process(y[:, 300:])
    for k in range(C_):
        cat = np.concatenate([q[k] for q in parts] + [rest[k]])
        assert np.array_equal(_bits(cat), _bits(one[k]))
    # random splits, different per channel, with a clone mid-stream
    rng = np.random.default_rng(L)
    p = sdr.Rrb(h, Is, Ds)
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
    p = sdr.Rrb(h, Is, Ds)
    first = p.process(y[:, :7])
    restm = np.ascontiguousarray(y[:, 7:])
    n = np.full(C_, restm.shape[1], np.uintp)
    need = p.output_count(restm.shape[1])
    cap = int(need.max())
    out = np.empty((C_, cap), np.complex64)
    got = np.zeros(C_, np.uintp)
    rc = sdr.lib().sdr_rrb_process(p.h, restm.ctypes.data, n.ctypes.data, restm.shape[1], out.ctypes.data, cap - 1,
                                   cap, got.ctypes.data)
    assert rc == 104 and not got.any()
    d_in = torch.from_numpy(restm).to(dev)
    d_out = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_rrb_process_dev(p.h, d_in.data_ptr(), n.ctypes.data, restm.shape[1], d_out.data_ptr(), cap - 1,
                                       cap, got.ctypes.data)
    assert rc == 104 and not got.any()
    second = p.process(restm)
    for k in range(C_):
        assert np.array_equal(_bits(np.concatenate([first[k], second[k]])), _bits(one[k]))


def test_rrb_odd_strides_and_primed_shards(sdr):
    torch, dev = _torch()
    C_, L = 4, 1023
    Is, Ds = [4, 147, 75, 3], [25, 160, 64, 4]
    h = _taps(C_, L, Is, False, 11)
    step = math.lcm(*[d // math.gcd(i, d) for i, d in zip(Is, Ds)])  # 6400: cuts with s I_k = 0 (mod D_k)
    nf = 4 * step
    y = _rows(C_, nf, 12)
    one = sdr.Rrb(h, Is, Ds).process(y)
    # odd device strides give the host bits, and nothing past the counts is written
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = y
    d_y = torch.from_numpy(pad).to(dev)
    cap = max(o.size for o in one)
    d_out = torch.full((C_, cap + 3), float("nan"), dtype=torch.complex64, device=dev)
    got = sdr.Rrb(h, Is, Ds, stream=st).process_dev(d_y, nf, nf + 5, d_out, cap, cap + 3)
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    for k in range(C_):
        assert got[k] == one[k].size
        assert np.array_equal(_bits(out[k, :got[k]]), _bits(one[k])) and np.isnan(out[k, got[k]:]).all()
    # shards cut at multiples of `step`, primed with H frames (a multiple of step >= max ceil(L / I_k))
    need = max(-(-L // i) for i in Is)
    H = -(-need // step) * step
    for world in (2, 4):
        cuts = [nf * r // world for r in range(world + 1)]
        assert all(c % step == 0 for c in cuts)
        parts = [[] for _ in range(C_)]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            plo = max(0, lo - H)
            z = sdr.Rrb(h, Is, Ds).process(y[:, plo:hi])
            for k in range(C_):
                parts[k].append(z[k][(lo - plo) * Is[k] // Ds[k]:])
        for k in range(C_):
            assert np.array_equal(_bits(np.concatenate(parts[k])), _bits(one[k]))


@pytest.mark.parametrize("I,D,L", [(4, 25, 255), (147, 160, 3529), (1, 5, 64), (75, 64, 1201)])
def test_rrb_nan_poisons_exactly_its_outputs(sdr, I, D, L):
    C_ = 2
    h = _taps(C_, L, [I, I], False, 13)
    h[1][L // 2] = 0.0  # a zero tap is still multiplied
    nf = 4 * (-(-L // I)) + 4 * D
    y = _rows(C_, nf, 14)
    m = nf // 2
    y[1, m] = np.complex64(complex(np.nan, 0.0))
    clean = y.copy()
    clean[1, m] = 0
    z = sdr.Rrb(h, I, D).process(y)
    ref = sdr.Rrb(h, I, D).process(clean)
    marker = np.zeros(nf)
    marker[m] = 1.0
    hit = R.computed_f64(np.abs(h[1].astype(np.float64)) + 1.0, marker, I, D) != 0
    assert hit.any() and not hit.all()
    assert np.isnan(z[1][hit]).all()
    assert np.array_equal(_bits(z[1][~hit]), _bits(ref[1][~hit]))
    assert np.array_equal(_bits(z[0]), _bits(ref[0]))


@pytest.mark.parametrize("C_", [1, 1024])
def test_rrb_launch_count(sdr, C_):
    torch, dev = _torch()
    Is, Ds = _ratios(C_, 15)
    h = _taps(1, 97, [1], True, 16)
    b = sdr.Rrb(h, Is, Ds)
    n = 2000
    d_y = torch.randn((C_, n), dtype=torch.complex64, device=dev)
    cap = int(b.output_count(n).max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    before = sdr.kernel_launch_count()
    b.process_dev(d_y, n, n, d_z, cap, cap)
    assert sdr.kernel_launch_count() - before <= 2
    torch.cuda.synchronize()


def _cascade_f64(x, h, incs, D, F=0):
    """the down-converter's definition in f64 by overlap-add convolution: [C, n // D]"""
    n = x.size
    keep = (np.arange(n // D) + 1) * D - 1
    out = np.empty((len(incs), n // D), np.complex128)
    for k, inc in enumerate(incs):
        z = x * ddc_ref.rot(ddc_ref.phases(F, np.arange(n), inc))
        out[k] = scipy.signal.oaconvolve(z, np.asarray(h, np.float64))[:n][keep]
    return out


def test_ddc_to_rrb_chain(sdr):
    """sdr_ddc (u8, tcgen05 path, D = 8) -> rrb 4/25 on 2^24 samples, device-resident, against the f64 cascade"""
    torch, dev = _torch()
    n, D, Ld = 1 << 24, 8, 255
    freqs = [0.1, -0.27]
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0)
    I2, D2, L2 = 4, 25, 401
    hr = _taps(1, L2, [I2], True, 17)
    raw = gen.random_u8(2 * n, 18)
    st = torch.cuda.current_stream(dev)
    ddc = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    nf = n // D
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((2, nf), dtype=torch.complex64, device=dev)
    assert ddc.process_dev(d_in, n, d_y, nf, nf) == nf
    assert ddc.last_path == 2
    rrb = sdr.Rrb(hr, I2, D2, n_channels=2, stream=st)
    cap = R.released(nf, I2, D2)
    d_z = torch.empty((2, cap), dtype=torch.complex64, device=dev)
    assert list(rrb.process_dev(d_y, nf, nf, d_z, cap, cap)) == [cap, cap]
    torch.cuda.synchronize()
    z = d_z.cpu().numpy()
    x = O.unpack_u8iq(raw).astype(np.complex128)
    incs = [int(v) for v in ddc.phase_inc]
    y64 = _cascade_f64(x, hd, incs, D)
    del x
    # the down-converter's per-output bar, carried through one phase of the resampler's taps, plus the bank's bar
    ff = max(np.sqrt((hr[c::I2].astype(np.float64) ** 2).sum()) for c in range(I2))
    for k in range(2):
        z64 = np.concatenate([R.computed_f64(hr.astype(np.float64), y64[k], I2, D2,
                                             outputs=np.arange(a, min(a + 32768, cap))) for a in range(0, cap, 32768)])
        bar = 1e-5 * np.abs(y64[k]).max() * ff + _bar(z64)
        assert np.abs(z[k] - z64).max() <= bar, k


def test_fcfb_to_rrb_rows_pass_unchanged(sdr):
    """sdr_fcfb's mixed-rate rows of one call, with its counts and out_stride, go straight into the bank"""
    torch, dev = _torch()
    n, L = 1 << 18, 255
    ds = [8, 10, 40]
    freqs = [0.2, -0.1, 0.33]
    h = gen.lowpass_taps(L, 0.5 / 40, 1.0)
    x = gen.complex_noise(n, 19)
    st = torch.cuda.current_stream(dev)
    fb = sdr.Fcfb(h, freqs, 1.0, ds, "c64", stream=st)
    cnt = fb.output_count(n)
    stride = int(cnt.max()) + 3
    d_x = torch.from_numpy(x).to(dev)
    d_y = torch.zeros((3, stride), dtype=torch.complex64, device=dev)
    got = fb.process_dev(d_x, n, d_y, stride, stride)
    assert list(got) == list(cnt)
    Is, Ds = [3, 4, 147], [4, 5, 160]
    hr = _taps(3, 97, Is, False, 20)
    rb = sdr.Rrb(hr, Is, Ds, stream=st)
    zc = rb.output_count(got)
    cap = int(zc.max())
    d_z = torch.empty((3, cap + 1), dtype=torch.complex64, device=dev)
    zgot = rb.process_dev(d_y, got, stride, d_z, cap, cap + 1)
    torch.cuda.synchronize()
    assert list(zgot) == list(zc)
    yh = d_y.cpu().numpy()
    rows = [yh[k, :got[k]] for k in range(3)]
    host = sdr.Rrb(hr, Is, Ds).process(rows)
    z = d_z.cpu().numpy()
    for k in range(3):
        assert np.array_equal(_bits(z[k, :zgot[k]]), _bits(host[k]))
    _check_channels(host, hr, rows, Is, Ds, oracle=False)


def test_rrb_to_duc_chain(sdr):
    """rrb 75/64 -> sdr_duc (I = 8), device-resident, at the bank's out_stride"""
    torch, dev = _torch()
    C_, nf, I = 3, 1 << 16, 8
    h = _taps(1, 1201, [75], True, 21)
    y = _rows(C_, nf, 22)
    st = torch.cuda.current_stream(dev)
    rb = sdr.Rrb(h, 75, 64, n_channels=C_, stream=st)
    cap = R.released(nf, 75, 64)
    stride = cap + 5
    d_y = torch.from_numpy(y).to(dev)
    d_z = torch.zeros((C_, stride), dtype=torch.complex64, device=dev)
    assert list(rb.process_dev(d_y, nf, nf, d_z, cap, stride)) == [cap] * C_
    hd = (I * gen.lowpass_taps(127, 0.5 / I, 1.0)).astype(np.float32)
    freqs = [-0.3, 0.05, 0.27]
    d_x = torch.empty(cap * I, dtype=torch.complex64, device=dev)
    assert sdr.Duc(hd, freqs, 1.0, I, stream=st).process_dev(d_z, cap, d_x, cap * I, stride) == cap * I
    torch.cuda.synchronize()
    z = sdr.Rrb(h, 75, 64, n_channels=C_).process(y)
    x = sdr.Duc(hd, freqs, 1.0, I).process(np.stack(z))
    assert np.array_equal(_bits(d_x.cpu().numpy()), _bits(x))
    _check_channels(z, h, y, [75] * C_, [64] * C_, oracle=False)


def test_rrb_spot_outputs_at_2_26(sdr):
    torch, dev = _torch()
    C_, I, D, L = 2, 147, 160, 147 * 24 + 1
    h = _taps(1, L, [I], True, 23)
    nout = 1 << 25
    nf = -(-nout * D // I)
    g = torch.Generator(device=dev).manual_seed(5)
    d_y = torch.randn((C_, nf), dtype=torch.complex64, device=dev, generator=g)
    cap = R.released(nf, I, D)
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    st = torch.cuda.current_stream(dev)
    assert list(sdr.Rrb(h, I, D, n_channels=C_, stream=st).process_dev(d_y, nf, nf, d_z, cap, cap)) == [cap] * C_
    torch.cuda.synchronize()
    for k in range(C_):
        for r0 in (0, cap // 3 + 77, cap - 4096):
            r = np.arange(r0, r0 + 4096)
            f0 = max(0, (r0 + 1) * D // I - L // I - 2)
            f1 = (r[-1] + 1) * D // I + 1
            yk = d_y[k, f0:f1].cpu().numpy().astype(np.complex128)
            # the f64 chain on frames f0 .. f1 - 1
            t1 = (r + 1) * D
            q, c = t1 // I, t1 % I
            i = np.arange(-(-L // I))
            tap = c[:, None] + i[None, :] * I
            j = q[:, None] - 1 - i[None, :] - f0
            ok = (tap < L) & (j + f0 >= 0)  # frames before the stream are 0
            hh = h.astype(np.float64)
            z64 = (np.where(ok, hh[np.minimum(tap, L - 1)], 0) * np.where(ok, yk[np.clip(j, 0, yk.size - 1)], 0)).sum(1)
            got = d_z[k, r0:r0 + 4096].cpu().numpy()
            assert np.abs(got - z64).max() <= _bar(z64), (k, r0)
    del d_y, d_z


def test_rrb_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "rrb_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "RRB MIRROR OK" in r.stdout, r.stdout + r.stderr

"""Fast-convolution channel bank (sdr_fcfb): every channel against f64 truth (mix with exact 64-bit phases, filter,
decimate by its own D_k) and against the crate's composition through the CPU oracle; agreement with sdr_ddc and
sdr_fir; a tone known answer; the round-off bound in terms of ||h_k|| and the block rms; a product-size run; 64-bit
stream positions; bit-identity across blockings, clones, resets, retries, addresses and block-aligned shards; NaN
poisoning of exactly the spanned blocks; draining; the C++ mirror."""
import ctypes as C_
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import signal as S

import ddc_ref as R
import fcfb_ref as Q
import gen

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATE = 2.4e6


def _input(fmt, n, seed):
    if fmt == "u8iq":
        import oracle_lib as O
        iq = gen.random_u8(2 * n, seed)
        return iq, O.unpack_u8iq(iq)
    x = gen.complex_noise(n, seed)
    return x, x


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(_bits(u), _bits(v)) for u, v in zip(a, b))


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _freqs(C, seed=0):
    rng = np.random.default_rng(seed + C)
    f = list(rng.uniform(-0.45, 0.45, C) * RATE)
    f[0] = 312.5e3
    if C > 1:
        f[1] = -687e3
    return f


def _taps(C, L, per_channel):
    if not per_channel:
        return gen.lowpass_taps(L, 100e3, RATE) if L > 1 else np.array([0.75], np.float32)
    return np.stack([gen.lowpass_taps(L, 60e3 + 10e3 * k, RATE) if L > 1 else np.array([0.5 + 0.1 * k], np.float32)
                     for k in range(C)])


def truth_f64(h, x, incs, ds, first=0, n_out=None):
    """the definition in f64 (fft convolution of the exactly mixed stream), channel k's first n_out[k] outputs"""
    x = np.asarray(x, np.complex128)
    n = x.size
    rows = []
    for k, (inc, d) in enumerate(zip(incs, ds)):
        z = x * R.rot(R.phases(first, np.arange(n), inc))
        hk = np.asarray(R.taps_of(h, k), np.float64)
        y = S.fftconvolve(z, hk)[:n] if hk.size > 1 else z * hk[0]
        keep = (np.arange(n // d) + 1) * d - 1
        rows.append(y[keep][:None if n_out is None else n_out[k]])
    return rows


def bar(N):
    return 2 * 1e-5 * math.log2(N)


def _check(got, truth, N, extra=0.0):
    for k, (g, t) in enumerate(zip(got, truth)):
        assert g.size <= t.size, k
        t = t[:g.size]
        if g.size == 0:
            continue
        assert np.abs(g - t).max() <= (bar(N) + extra) * np.abs(t).max(), k


DSETS = {"one": [1], "eight": [8], "ten": [10], "mixed": [1, 2, 8, 10, 40]}
LS = (1, 64, 255, 511, 512, 4095, 65537)
GRID = [(ds, L) for ds in DSETS for L in LS]


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("dset,L", GRID)
def test_fcfb_every_channel_against_f64_and_oracle(sdr, fmt, dset, L):
    i = GRID.index((dset, L))
    C = (1, 3, 8, 17)[i % 4]
    per_channel = bool((i // 4 + i) % 2)
    base = DSETS[dset]
    ds = [base[k % len(base)] for k in range(C)]
    h = _taps(C, L, per_channel)
    N, P = Q.geometry(L, ds)
    n = 3 * N + 1000 + 37
    raw, x = _input(fmt, n, 40 + L + i)
    b = sdr.Fcfb(h, _freqs(C, i), RATE, ds, fmt)
    assert b.geometry == (N, P)
    got = b.process(raw)
    incs = list(b.phase_inc)
    want = Q.counts(n, ds, P, Q.off0(0, ds, P))
    assert [g.size for g in got] == want
    _check(got, truth_f64(h, x, incs, ds), N)
    if L <= 4095:  # the oracle's direct-form FIR: n L multiply-adds on the CPU
        oracle = [R.oracle_f32(R.taps_of(h, k), x, [incs[k]], ds[k])[0] for k in range(C)]
        _check(got, oracle, N, 1e-5)
    if len(set(ds)) == 1:
        # the same function as sdr_ddc: agree within both bars
        dd = sdr.Ddc(h, _freqs(C, i), RATE, ds[0], fmt).process(raw)
        _check(got, list(dd), N, 1e-5)


@pytest.mark.parametrize("fmt,D,L", [("c64", 1, 4095), ("u8iq", 10, 255), ("c64", 8, 64)])
def test_fcfb_single_channel_at_zero_frequency_equals_fir(sdr, fmt, D, L):
    h = gen.lowpass_taps(L, 100e3, RATE)
    n = 200000 + 3
    raw, _ = _input(fmt, n, 9)
    got = sdr.Fcfb(h, [0.0], RATE, D, fmt).process(raw)[0]
    want = sdr.Fir(h, fmt, decimation=D).process(raw)
    N, _ = sdr.fcfb_geometry(L, [D])
    assert np.abs(got - want[:got.size]).max() <= (bar(N) + 1e-5) * np.abs(want).max()


def test_fcfb_tone_lands_in_its_channel(sdr):
    L = 255
    h = gen.lowpass_taps(L, 100e3, RATE)
    freqs = [312.5e3, -687e3, 900e3, 312.5e3]
    ds = [8, 10, 16, 4]
    delta, A = 23e3, 0.4
    n = 1 << 16
    raw = gen.tone_noise_u8(n, RATE, freqs[0] + delta, A, 0.0, 3)
    y = sdr.Fcfb(h, freqs, RATE, ds, "u8iq").process(raw)
    H = abs(np.sum(h.astype(np.float64) * np.exp(-2j * np.pi * delta / RATE * np.arange(L))))
    for k in (0, 3):
        s = y[k][2 * L // ds[k]:]
        assert np.allclose(np.abs(s), A * H, rtol=0.02)
        dphi = np.angle(s[1:] * np.conj(s[:-1]))
        assert np.allclose(dphi, 2 * np.pi * delta * ds[k] / RATE, atol=0.02)
    for k in (1, 2):  # 400 kHz and more away: stop band
        assert np.abs(y[k][2 * L // ds[k]:]).max() <= 0.02 * A


def test_fcfb_round_off_follows_block_power(sdr):
    """a channel holding only noise 60 dB below an out-of-band tone: the error follows ||h_k||_2 rms(block), not the
    channel's own level (DESIGN.md K9): |y - y_f64| <= 8 eps log2(N) ||h_k||_2 rms, eps = 2^-24"""
    L, D = 1023, 8
    h = gen.lowpass_taps(L, 50e3, RATE)
    n = 1 << 18
    t = np.arange(n)
    rng = np.random.default_rng(5)
    tone = 0.9 * np.exp(2j * np.pi * 700e3 / RATE * t)
    noise = 0.9e-3 / math.sqrt(2) * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    x = (tone + noise).astype(np.complex64)
    freqs = [-300e3, 700e3]
    b = sdr.Fcfb(h, freqs, RATE, D, "c64")
    N, _ = b.geometry
    got = b.process(x)
    truth = truth_f64(h, x, list(b.phase_inc), [D, D])
    rms = math.sqrt(np.mean(np.abs(x.astype(np.complex128)) ** 2))
    hn = float(np.linalg.norm(h.astype(np.float64)))
    bound = 8 * 2.0 ** -24 * math.log2(N) * hn * rms
    err = np.abs(got[0] - truth[0][:got[0].size]).max()
    assert err <= bound, (err, bound)
    # the channel still sees its own noise floor: the error is well below it
    assert err <= 0.05 * np.abs(truth[0]).std()
    # and the tone channel meets the per-channel bar
    _check(got[1:], truth[1:], N)


def test_fcfb_product_size(sdr):
    torch, dev = _torch()
    import oracle_lib as O
    n, L = 1 << 26, 4095
    ds = [8, 8, 16, 16, 32, 32, 64, 64]
    C = len(ds)
    h = gen.lowpass_taps(L, 20e3, RATE)
    raw = gen.random_u8(2 * n, 77)
    st = torch.cuda.current_stream(dev)
    b = sdr.Fcfb(h, _freqs(C), RATE, ds, "u8iq", stream=st)
    cnt = b.output_count(n)
    d_in = torch.from_numpy(raw).to(dev)
    d_out = torch.empty((C, int(cnt.max())), dtype=torch.complex64, device=dev)
    got = b.process_dev(d_in, n, d_out, int(cnt.max()))
    torch.cuda.synchronize()
    assert list(got) == list(cnt)
    x = O.unpack_u8iq(raw)
    N, _ = b.geometry
    for k in range(C):
        nf = int(cnt[k])
        outs = np.unique(np.concatenate([np.arange(64), np.arange(nf // 2 - 7, nf // 2 + 100), np.arange(nf - 64, nf)]))
        row = d_out[k, torch.from_numpy(outs).to(dev)].cpu().numpy()
        truth = R.rotated_f64(h, x, [int(b.phase_inc[k])], ds[k], outputs=outs)[0]
        assert np.abs(row - truth).max() <= bar(N) * np.abs(truth).max(), k
    assert bool(torch.isfinite(torch.view_as_real(d_out)).all())


@pytest.mark.parametrize("first", [(1 << 40) + 12345, (1 << 63) - 7])
@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_fcfb_64_bit_stream_positions(sdr, first, fmt):
    ds, L = [8, 10, 1, 40], 255
    h = _taps(len(ds), L, True)
    n = 30000 + 11
    raw, x = _input(fmt, n, 31)
    b = sdr.Fcfb(h, _freqs(len(ds)), RATE, ds, fmt, first_sample=first)
    got = b.process(raw)
    N, P = b.geometry
    assert [g.size for g in got] == Q.counts(n, ds, P, Q.off0(first, ds, P))
    _check(got, truth_f64(h, x, list(b.phase_inc), ds, first), N)


def _pieces(n, seed, P):
    rng = np.random.default_rng(seed)
    cuts = set(rng.choice(np.arange(1, n), 9, replace=False).tolist())
    cuts |= {1, 2, 3, P - 1, P, 2 * P + 1}  # 1-sample calls, calls that end mid-block and on a block end
    cuts = sorted(c for c in cuts if 0 < c < n)
    return [0] + cuts + [n]


def _cat(parts, C):
    return [np.concatenate([p[k] for p in parts]) for k in range(C)]


@pytest.mark.parametrize("fmt,ds,L,first", [("u8iq", [8, 10, 1, 40, 2], 255, 999), ("c64", [8], 4095, 0),
                                            ("c64", [1, 3], 64, 12345), ("u8iq", [16, 16, 32], 511, 7)])
def test_fcfb_blocking_clone_reset_are_bit_exact(sdr, fmt, ds, L, first):
    C = len(ds)
    h = _taps(C, L, True)
    b = sdr.Fcfb(h, _freqs(C), RATE, ds, fmt, first_sample=first)
    N, P = b.geometry
    n = 5 * N + 3
    raw, _ = _input(fmt, n, 5)
    per = 2 if fmt == "u8iq" else 1
    one = b.process(raw)
    b.reset()
    p = _pieces(n, L, P)
    parts = []
    mid = p[len(p) // 2]
    for a, e in zip(p[:-1], p[1:]):
        parts.append(b.process(raw[per * a:per * e]))
        if a == mid:
            clone = b.clone()
            cut = e
    assert _same(_cat(parts, C), one)
    rest = clone.process(raw[per * cut:])
    assert _same(rest, [o[o.size - r.size:] for o, r in zip(one, rest)])
    b.reset()
    assert _same(b.process(raw), one)


def test_fcfb_too_small_output_is_refused_without_state_change(sdr):
    torch, dev = _torch()
    ds, L = [8, 10, 1], 127
    C = len(ds)
    h = _taps(C, L, False)
    n = 20000
    raw, _ = _input("u8iq", n, 8)
    one = sdr.Fcfb(h, _freqs(C), RATE, ds).process(raw)
    b = sdr.Fcfb(h, _freqs(C), RATE, ds)
    first = b.process(raw[:2 * 1001])
    rest = np.ascontiguousarray(raw[2 * 1001:])
    n_rest = rest.size // 2
    need = int(b.output_count(n_rest).max())
    out = np.empty((C, need), np.complex64)
    got = np.full(C, 7, np.uintp)
    assert sdr.lib().sdr_fcfb_process(b.h, rest.ctypes.data, n_rest, out.ctypes.data, need - 1, need,
                                      got.ctypes.data) == 104
    assert (got == 0).all()
    d_in = torch.from_numpy(rest).to(dev)
    d_out = torch.empty((C, need), dtype=torch.complex64, device=dev)
    assert sdr.lib().sdr_fcfb_process_dev(b.h, d_in.data_ptr(), n_rest, d_out.data_ptr(), need - 1, need,
                                          got.ctypes.data) == 104
    assert int(b.output_count(n_rest).max()) == need
    second = b.process(rest)
    assert _same(_cat([first, second], C), one)


def test_fcfb_u8_at_odd_element_offsets(sdr):
    torch, dev = _torch()
    ds, L = [8, 10], 255
    h = _taps(2, L, True)
    n = 50000
    raw, _ = _input("u8iq", n, 12)
    one = sdr.Fcfb(h, _freqs(2), RATE, ds).process(raw)
    st = torch.cuda.current_stream(dev)
    for pad in (1, 3, 7):
        d_raw = torch.from_numpy(np.concatenate([np.zeros(2 * pad, np.uint8), raw])).to(dev)
        b = sdr.Fcfb(h, _freqs(2), RATE, ds, stream=st)
        cnt = b.output_count(n)
        d_out = torch.empty((2, int(cnt.max())), dtype=torch.complex64, device=dev)
        got = b.process_dev(d_raw.data_ptr() + 2 * pad, n, d_out, int(cnt.max()))
        torch.cuda.synchronize()
        rows = [d_out[k, :int(got[k])].cpu().numpy() for k in range(2)]
        assert _same(rows, one)


@pytest.mark.parametrize("fmt,ds", [("u8iq", [8, 10, 40]), ("c64", [1, 2])])
def test_fcfb_shards_concatenate_to_one_stream(sdr, fmt, ds):
    """shards cut on block boundaries of the absolute grid, halo = N - P rounded up to a multiple of Dl, first_sample =
    the halo start, give the bits of one call"""
    torch, dev = _torch()
    C, L = len(ds), 255
    h = _taps(C, L, True)
    first = 3 * Q.lcm_of(ds) + 1   # eps != 0
    N, P = Q.geometry(L, ds)
    Dl = Q.lcm_of(ds)
    o0 = Q.off0(first, ds, P)
    n = 40 * P + 17
    raw, _ = _input(fmt, n, 17)
    per = 2 if fmt == "u8iq" else 1
    es = 2 if fmt == "u8iq" else 8
    one = sdr.Fcfb(h, _freqs(C), RATE, ds, fmt, first_sample=first).process(raw)
    halo = -(-(N - P) // Dl) * Dl
    st = torch.cuda.current_stream(dev)
    d_raw = torch.from_numpy(raw).to(dev)
    for world in (2, 3):
        # block boundaries in handle coordinates: j P - o0
        cuts = [0] + [(j * 40 // world) * P - o0 for j in range(1, world)] + [n]
        parts = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            hlo = max(0, lo - halo)
            b = sdr.Fcfb(h, _freqs(C), RATE, ds, fmt, first_sample=first + hlo, stream=st)
            cnt = b.output_count(hi - hlo)
            d_out = torch.empty((C, max(int(cnt.max()), 1)), dtype=torch.complex64, device=dev)
            got = b.process_dev(d_raw.data_ptr() + hlo * es, hi - hlo, d_out, max(int(cnt.max()), 1))
            torch.cuda.synchronize()
            rows = []
            for k, d in enumerate(ds):
                skip = (lo - hlo) // d  # outputs before the cut belong to the previous shard
                rows.append(d_out[k, skip:int(got[k])].cpu().numpy())
            parts.append(rows)
        cat = _cat(parts, C)
        # the last shard releases the same blocks as the one-call handle
        assert _same(cat, one)


@pytest.mark.parametrize("ds,L", [([8, 10, 1], 255), ([40], 1000)])
def test_fcfb_nan_poisons_exactly_its_blocks(sdr, ds, L):
    b = sdr.Fcfb(gen.lowpass_taps(L, 100e3, RATE), _freqs(len(ds)), RATE, ds, "c64", first_sample=5)
    N, P = b.geometry
    o0 = Q.off0(5, ds, P)
    n = 8 * N + 100
    x = gen.complex_noise(n, 2)
    clean = b.clone().process(x)
    s = n // 2 + 3
    x[s] = np.complex64(complex(np.nan, 0.0))
    y = b.process(x)
    for k, d in enumerate(ds):
        m = np.arange(y[k].size)
        e = (m + 1) * d - 1                      # newest sample of each output (handle index)
        j = (e + o0) // P                         # its block
        span_lo = (j + 1) * P - o0 - N
        hit = (span_lo <= s) & (s < span_lo + N)
        assert hit.sum() >= 1
        assert np.isnan(y[k][hit]).all()
        assert np.array_equal(_bits(y[k][~hit]), _bits(clean[k][~hit]))


def test_fcfb_drain_with_n_zeros(sdr):
    ds, L = [8, 10, 1], 511
    h = _taps(3, L, True)
    n = 12345
    raw, x = _input("c64", n, 21)
    b = sdr.Fcfb(h, _freqs(3), RATE, ds, "c64")
    N, _ = b.geometry
    y = b.process(raw)
    tail = b.process(np.zeros(N, np.complex64))
    full = [np.concatenate([a, t])[:n // d] for a, t, d in zip(y, tail, ds)]
    assert [f.size for f in full] == [n // d for d in ds]
    _check(full, truth_f64(h, x, list(b.phase_inc), ds), N)


def test_fcfb_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "fcfb_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "FCFB MIRROR OK" in r.stdout, r.stdout + r.stderr

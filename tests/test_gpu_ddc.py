"""Digital down-converter bank (sdr_ddc): every channel against f64 truth (mix with exact 64-bit phases, filter,
decimate) and against the crate's own composition through the CPU oracle, on both kernels; product size on the tensor
path; a tone known answer; agreement with sdr_pfb; streaming, clone / reset, sharding and 64-bit phase positions;
NaN window bounds; PllBatch fed from the channel-major rows; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import ddc_ref as R
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


def _tc_expected(fmt, general, D, L):
    """the tensor path's geometry (ddc.cu ddc_tc_geometry) for one channel"""
    if fmt != "u8iq" or general or 32 % D or L > 511:
        return False
    PC = 32 // D
    KS = (L + 7 + 32 - D + 15) // 16
    Ng = -(-(6 * PC) // 16) * 16
    stage = (64 * 127 + 32 * KS + 1023) // 1024 * 1024
    return KS * Ng * 32 + 2 * stage + 1280 <= 220 * 1024


def _check(got, truth, oracle=None):
    for k in range(truth.shape[0]):
        bar = 1e-5 * np.abs(truth[k]).max()
        assert np.abs(got[k] - truth[k]).max() <= bar, k
        if oracle is not None:
            assert np.abs(got[k] - oracle[k]).max() <= bar, k


CASES = [(D, L) for D in (1, 2, 8, 10, 16, 32) for L in (1, 64, 255, 511)]


@pytest.mark.parametrize("fmt,general", [("u8iq", False), ("u8iq", True), ("c64", False)])
@pytest.mark.parametrize("D,L", CASES + [(8, 1000), (3, 1000)])
def test_ddc_every_channel_against_f64_and_oracle(sdr, fmt, general, D, L):
    i = CASES.index((D, L)) if (D, L) in CASES else 1
    C = (1, 3, 8, 17)[i % 4]
    per_channel = bool((i // 4 + i) % 2)
    h = _taps(C, L, per_channel)
    n = max(3000, 3 * L + 64 * D) + 37
    raw, x = _input(fmt, n, 40 + D + L)
    freqs = _freqs(C, D)
    d = sdr.Ddc(h, freqs, RATE, D, fmt, general=general)
    got = d.process(raw)
    assert got.shape == (C, n // D)
    assert d.last_path == (2 if _tc_expected(fmt, general, D, L) else 1)
    incs = list(d.phase_inc)
    truth = R.mix_first_f64(np.asarray(h, np.float64), x, incs, D)
    oracle = R.oracle_f32(h, x, incs, D)
    _check(got, truth, oracle)


def test_ddc_product_size_on_the_tensor_path(sdr):
    torch, dev = _torch()
    n, C, D, L = 1 << 26, 8, 8, 255
    h = gen.lowpass_taps(L, 100e3, RATE)
    raw = gen.random_u8(2 * n, 77)
    import oracle_lib as O
    st = torch.cuda.current_stream(dev)
    d = sdr.Ddc(h, _freqs(C), RATE, D, "u8iq", stream=st)
    d_in = torch.from_numpy(raw).to(dev)
    nf = n // D
    d_out = torch.empty((C, nf), dtype=torch.complex64, device=dev)
    assert d.process_dev(d_in, n, d_out, nf) == nf
    torch.cuda.synchronize()
    assert d.last_path == 2
    outs = np.unique(np.concatenate([np.arange(64), np.arange(nf // 2 - 7, nf // 2 + 300), np.arange(nf - 64, nf)]))
    got = d_out[:, torch.from_numpy(outs).to(dev)].cpu().numpy()
    x = O.unpack_u8iq(raw)
    truth = R.rotated_f64(h, x, list(d.phase_inc), D, outputs=outs)
    _check(got, truth)
    assert bool(torch.isfinite(torch.view_as_real(d_out)).all())


@pytest.mark.parametrize("general", [False, True])
def test_ddc_tone_lands_in_its_channel(sdr, general):
    D, L = 8, 255
    h = gen.lowpass_taps(L, 100e3, RATE)
    freqs = [312.5e3, -687e3, 900e3]
    delta, A = 23e3, 0.4
    n = 1 << 16
    raw = gen.tone_noise_u8(n, RATE, freqs[0] + delta, A, 0.0, 3)
    y = sdr.Ddc(h, freqs, RATE, D, "u8iq", general=general).process(raw)
    H = abs(np.sum(h.astype(np.float64) * np.exp(-2j * np.pi * delta / RATE * np.arange(L))))
    s = y[0, 2 * L // D:]
    assert np.allclose(np.abs(s), A * H, rtol=0.02)
    dphi = np.angle(s[1:] * np.conj(s[:-1]))
    assert np.allclose(dphi, 2 * np.pi * delta * D / RATE, atol=0.02)
    for k in (1, 2):  # 400 kHz and more away: stop band
        assert np.abs(y[k, 2 * L // D:]).max() <= 0.02 * A


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("general", [False, True])
def test_ddc_agrees_with_pfb(sdr, fmt, general):
    M, D, L = 16, 8, 255
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    n = 40000 + 5
    raw, _ = _input(fmt, n, 21)
    pfb = sdr.Pfb(h, M, D, fmt, channel_major=True).process(raw)
    d = sdr.Ddc(h, [k / M for k in range(M)], 1.0, D, fmt, general=general)
    assert [int(v) for v in d.phase_inc] == [(k << 64) // M for k in range(M)]
    y = d.process(raw)
    N = (np.arange(n // D) + 1) * D - 1
    want = np.exp(-2j * np.pi * np.outer(np.arange(M), N % M) / M) * pfb
    bar = 1e-5 * np.log2(M) * np.abs(want).max()
    assert np.abs(y - want).max() <= bar


def _pieces(n, seed):
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.choice(np.arange(1, n), 9, replace=False))
    return np.concatenate([[0], cuts, [n]])


@pytest.mark.parametrize("fmt,general,D,L", [("u8iq", False, 8, 255), ("u8iq", False, 1, 64), ("u8iq", False, 32, 511),
                                             ("u8iq", True, 8, 255), ("c64", False, 10, 300), ("u8iq", False, 16, 97)])
def test_ddc_blocking_clone_reset_are_bit_exact(sdr, fmt, general, D, L):
    C = 5
    h = _taps(C, L, True)
    n = 60000 + 3
    raw, _ = _input(fmt, n, 5)
    per = 2 if fmt == "u8iq" else 1
    d = sdr.Ddc(h, _freqs(C), RATE, D, fmt, first_sample=999, general=general)
    one = d.process(raw)
    d.reset()
    p = _pieces(n, D + L)
    parts = []
    for a, b in zip(p[:-1], p[1:]):
        parts.append(d.process(raw[per * a:per * b]))
        if a == p[4]:
            clone = d.clone()
            cut = b
    assert np.array_equal(_bits(np.concatenate(parts, axis=1)), _bits(one))
    rest = clone.process(raw[per * cut:])
    assert np.array_equal(_bits(rest), _bits(one[:, one.shape[1] - rest.shape[1]:]))
    d.reset()
    assert np.array_equal(_bits(d.process(raw)), _bits(one))


@pytest.mark.parametrize("general", [False, True])
def test_ddc_too_small_output_is_refused_without_state_change(sdr, general):
    import ctypes as C_
    torch, dev = _torch()
    C, D, L = 3, 8, 127
    h = _taps(C, L, False)
    n = 20000
    raw, _ = _input("u8iq", n, 8)
    one = sdr.Ddc(h, _freqs(C), RATE, D, general=general).process(raw)
    d = sdr.Ddc(h, _freqs(C), RATE, D, general=general)
    first = d.process(raw[:2 * 1001])
    rest = np.ascontiguousarray(raw[2 * 1001:])
    n_rest = rest.size // 2
    need = d.output_count(n_rest)
    out = np.empty((C, need), np.complex64)
    got = C_.c_size_t(0)
    assert sdr.lib().sdr_ddc_process(d.h, rest.ctypes.data, n_rest, out.ctypes.data, need - 1, need, C_.byref(got)) == 104
    assert got.value == 0
    d_in = torch.from_numpy(rest).to(dev)
    d_out = torch.empty((C, need), dtype=torch.complex64, device=dev)
    assert sdr.lib().sdr_ddc_process_dev(d.h, d_in.data_ptr(), n_rest, d_out.data_ptr(), need - 1, need,
                                         C_.byref(got)) == 104
    assert d.output_count(n_rest) == need
    second = d.process(rest)
    assert np.array_equal(_bits(np.concatenate([first, second], axis=1)), _bits(one))


@pytest.mark.parametrize("fmt,general,D", [("u8iq", False, 8), ("u8iq", False, 16), ("u8iq", True, 10),
                                           ("c64", False, 8)])
def test_ddc_shards_concatenate_to_one_stream(sdr, fmt, general, D):
    """halo shards (cuts on multiples of D, first_sample = the halo start) of a stream that starts 3 samples into its
    buffer, so that no shard's first sample is 16-byte aligned, give the bits of one call on an aligned copy"""
    torch, dev = _torch()
    from sdr_b200 import shard
    n, C, L, pad = 1 << 21, 4, 255, 3
    h = _taps(C, L, True)
    raw, _ = _input(fmt, n, 17)
    es = 2 if fmt == "u8iq" else 8
    per = 2 if fmt == "u8iq" else 1
    st = torch.cuda.current_stream(dev)
    d_raw = torch.from_numpy(np.concatenate([np.zeros(per * pad, raw.dtype), raw])).to(dev)
    base = d_raw.data_ptr() + pad * es
    nf = n // D
    one = sdr.Ddc(h, _freqs(C), RATE, D, fmt, general=general).process(raw)
    assert one.shape == (C, nf)
    halo = -(-(L - 1) // D) * D
    for world in (1, 2, 3):
        parts = []
        for rank in range(world):
            lo, hi, hlo = shard.sample_range(n, world, rank, halo=halo, align=D)
            d = sdr.Ddc(h, _freqs(C), RATE, D, fmt, first_sample=hlo, general=general, stream=st)
            cnt = d.output_count(hi - hlo)
            d_out = torch.empty((C, max(cnt, 1)), dtype=torch.complex64, device=dev)
            assert (base + hlo * es) % 16 != 0
            got = d.process_dev(base + hlo * es, hi - hlo, d_out, cnt)
            torch.cuda.synchronize()
            parts.append(d_out.cpu().numpy()[:, (lo - hlo) // D:got])
        cat = np.concatenate(parts, axis=1)
        assert cat.shape == one.shape
        assert np.array_equal(_bits(cat), _bits(one))


@pytest.mark.parametrize("first", [(1 << 40) + 12345, (1 << 63) - 7])
@pytest.mark.parametrize("fmt,general", [("u8iq", False), ("u8iq", True), ("c64", False)])
def test_ddc_64_bit_stream_positions(sdr, first, fmt, general):
    C, D, L = 4, 8, 255
    h = _taps(C, L, True)
    n = 30000 + 11
    raw, x = _input(fmt, n, 31)
    d = sdr.Ddc(h, _freqs(C), RATE, D, fmt, first_sample=first, general=general)
    got = d.process(raw)
    truth = R.mix_first_f64(np.asarray(h, np.float64), x, list(d.phase_inc), D, first)
    _check(got, truth)


@pytest.mark.parametrize("D,L", [(8, 255), (10, 67), (1, 1000)])
def test_ddc_nan_poisons_exactly_its_windows(sdr, D, L):
    n = 20 * L + 100
    x = gen.complex_noise(n, 2)
    s = n // 2 + 3
    x[s] = np.complex64(complex(np.nan, 0.0))
    y = sdr.Ddc(gen.lowpass_taps(L, 100e3, RATE), _freqs(3), RATE, D, "c64").process(x)
    e = (np.arange(y.shape[1]) + 1) * D - 1
    hit = (e >= s) & (e - L + 1 <= s)
    assert hit.sum() >= 1
    assert np.isnan(y[:, hit]).all()
    assert np.isfinite(y[:, ~hit]).all()


def test_ddc_channel_major_rows_feed_pll_batch(sdr):
    torch, dev = _torch()
    C, D = 4, 8
    h = gen.lowpass_taps(255, 100e3, RATE)
    n = 4096 * D
    freqs = [312.5e3, -687e3, 100e3, 0.0]
    raw = gen.tone_noise_u8(n, RATE, freqs[0] + 2e3, 0.5, 0.05, 5)
    d = sdr.Ddc(h, freqs, RATE, D)
    y = d.process(raw)
    nf = y.shape[1]
    design = sdr.PllDesign(0.0, 0.035, sdr.BiquadD.LowPass(8e3, .7), sdr.Identity(), sdr.Identity())
    want_v, want_l = sdr.PllBatch([design], C, RATE / D).process(np.ascontiguousarray(y))
    st = torch.cuda.current_stream(dev)
    stride = nf + 3
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((C, stride), dtype=torch.complex64, device=dev)
    assert sdr.Ddc(h, freqs, RATE, D, stream=st).process_dev(d_in, n, d_y, nf, stride) == nf
    d_v = torch.empty((C, nf), dtype=torch.float32, device=dev)
    d_l = torch.empty((C, nf), dtype=torch.uint8, device=dev)
    sdr.PllBatch([design], C, RATE / D, stream=st).process_dev(d_y, nf, d_v, d_l, in_stride=stride, out_stride=nf)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(d_v.cpu().numpy()), _bits(want_v))
    assert np.array_equal(d_l.cpu().numpy(), want_l)


def test_ddc_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "ddc_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DDC MIRROR OK" in r.stdout, r.stdout + r.stderr

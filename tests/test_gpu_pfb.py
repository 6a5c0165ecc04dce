"""Polyphase filter bank (sdr_pfb): every channel against the crate's own composition -- Fir(h e^{+2 pi i k n / M})
followed by Decimate(D), through the CPU oracle -- and against f64 truth; layout flags, streaming, sharding, window
bounds, both front-end kernels and interoperation with PllBatch."""
import os
import subprocess

import numpy as np
import pytest

import gen
import oracle_lib as O
import pfb_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bar(M, y64):
    """the FFT bar of DESIGN.md section 4: 1e-5 log2(M) of max|y|"""
    return 1e-5 * max(1.0, np.log2(M)) * np.abs(y64).max()


def _input(fmt, n, seed):
    """(raw input for the bank, its c64 values)"""
    if fmt == "u8iq":
        iq = gen.random_u8(2 * n, seed)
        return iq, O.unpack_u8iq(iq)
    x = gen.complex_noise(n, seed)
    return x, x


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("M", [8, 16])
@pytest.mark.parametrize("Dsel", ["M", "M/2", 3])
def test_pfb_pinned_to_fir_decimate(sdr, fmt, M, Dsel):
    D = {"M": M, "M/2": M // 2}.get(Dsel, Dsel)
    L = 6 * M + 5
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    raw, x = _input(fmt, 3000, 40 + M + D)
    got = sdr.Pfb(h, M, D, fmt).process(raw)
    truth = R.direct_f64(h.astype(np.float64), x, M, D)
    oracle = R.direct_oracle_f32(h, x, M, D)
    assert got.shape == truth.shape == oracle.shape == (3000 // D, M)
    bar = _bar(M, truth)
    assert np.abs(got - truth).max() <= bar
    assert np.abs(got - oracle).max() <= bar


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("M,D", [(64, 64), (64, 32), (1024, 1024), (1024, 512), (4096, 4096), (4096, 2048),
                                 (1000, 1000), (1000, 500)])
def test_pfb_product_sizes_against_f64(sdr, fmt, M, D):
    n = 1 << 20
    h = gen.lowpass_taps(16 * M, 0.5 / M, 1.0)
    raw, x = _input(fmt, n, 7 + M + D)
    got = sdr.Pfb(h, M, D, fmt).process(raw)
    nf = n // D
    assert got.shape == (nf, M)
    frames = np.unique(np.concatenate([np.arange(min(nf, 48)), np.arange(nf // 2, nf // 2 + 16), np.arange(nf - 48, nf)]))
    truth = R.polyphase_f64(h, x, M, D, frames=frames)
    assert np.abs(got[frames] - truth).max() <= _bar(M, truth)
    assert np.isfinite(got).all()


@pytest.mark.parametrize("M,D,k0", [(64, 32, 5), (64, 64, 50), (1024, 512, 300)])
def test_pfb_tone_lands_in_its_channel(sdr, M, D, k0):
    L = 16 * M
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    n = 40 * L
    A = 0.5
    t = np.arange(n, dtype=np.float64)
    x = (A * np.exp(2j * np.pi * k0 / M * t)).astype(np.complex64)
    y = sdr.Pfb(h, M, D, "c64").process(x)
    ys = sdr.Pfb(h, M, D, "c64", shift=True).process(x)
    first = -(-(L - 1 + 1) // D)  # frames whose window lies inside the signal: (m+1) D - 1 >= L - 1
    y, ys = y[first:], ys[first:]
    h64 = h.astype(np.float64)
    gain = abs(h64.sum())
    bar = _bar(M, A * gain * np.ones(1))
    assert np.abs(np.abs(y[:, k0]) - A * gain).max() <= bar
    # stop-band level of the prototype: max |H(nu)| for 2/M <= |nu| <= 1/2, from h in f64
    nfft = 64 * L
    H = np.abs(np.fft.fft(h64, nfft))  # h real: |H(-nu)| = |H(nu)|
    stop = 1.01 * H[int(np.ceil(2.0 / M * nfft)):nfft // 2 + 1].max()
    far = [k for k in range(M) if min((k - k0) % M, (k0 - k) % M) >= 2]
    assert np.abs(y[:, far]).max() <= A * stop + bar
    assert np.argmax(np.abs(ys).mean(axis=0)) == (k0 + M // 2) % M
    assert np.abs(np.abs(ys[:, (k0 + M // 2) % M]) - A * gain).max() <= bar


@pytest.mark.parametrize("M,D,fmt", [(16, 5, "c64"), (1024, 512, "u8iq"), (1000, 1000, "c64")])
def test_pfb_layout_flags_are_exact(sdr, M, D, fmt):
    torch, dev = _torch()
    h = gen.lowpass_taps(8 * M + 3, 0.5 / M, 1.0)
    n = 200 * D + 7
    raw, _ = _input(fmt, n, 3)
    plain = sdr.Pfb(h, M, D, fmt).process(raw)
    nf = plain.shape[0]
    shifted = sdr.Pfb(h, M, D, fmt, shift=True).process(raw)
    perm = (np.arange(M) - M // 2) % M
    assert np.array_equal(_bits(shifted), _bits(plain[:, perm]))
    cm_host = sdr.Pfb(h, M, D, fmt, channel_major=True).process(raw)
    assert np.array_equal(_bits(cm_host), _bits(plain.T))
    # device entry points: channel-major rows with a stride beyond the frame count, frame-major with a padded stride
    st = torch.cuda.current_stream(dev)
    d_in = torch.from_numpy(np.ascontiguousarray(raw)).to(dev)
    stride = nf + 5
    d_cm = torch.full((M, stride), float("nan"), dtype=torch.complex64, device=dev)
    got = sdr.Pfb(h, M, D, fmt, channel_major=True, stream=st).process_dev(d_in, n, d_cm, nf, stride)
    d_fm = torch.full((nf, M + 3), float("nan"), dtype=torch.complex64, device=dev)
    got2 = sdr.Pfb(h, M, D, fmt, stream=st).process_dev(d_in, n, d_fm, nf, M + 3)
    torch.cuda.synchronize()
    assert got == got2 == nf
    cm = d_cm.cpu().numpy()
    fm = d_fm.cpu().numpy()
    assert np.array_equal(_bits(cm[:, :nf]), _bits(plain.T)) and np.isnan(cm[:, nf:]).all()
    assert np.array_equal(_bits(fm[:, :M]), _bits(plain)) and np.isnan(fm[:, M:]).all()


@pytest.mark.parametrize("M,D,L,fmt", [(64, 48, 1000, "c64"), (256, 128, 16 * 256, "u8iq"), (1000, 1000, 16000, "c64")])
def test_pfb_streaming(sdr, M, D, L, fmt):
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    n = 60 * D + 13
    raw, _ = _input(fmt, n, 9)
    per = 2 if fmt == "u8iq" else 1
    one = sdr.Pfb(h, M, D, fmt).process(raw)
    p = sdr.Pfb(h, M, D, fmt)
    parts, pos = [], 0
    blocks = [1, 1, D - 1, 0, D // 2, 3 * D + 1, 1, 0, 7 * D - 3]
    blocks.append(n - sum(blocks))
    clone = None
    for i, b in enumerate(blocks):
        parts.append(p.process(raw[per * pos:per * (pos + b)]))
        pos += b
        if i == 5:
            clone = p.clone()
            rest = raw[per * pos:]
    assert pos == n
    assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
    # a clone taken mid-stream continues like the original
    cont = clone.process(rest)
    assert np.array_equal(_bits(cont), _bits(one[one.shape[0] - cont.shape[0]:]))
    # reset equals a fresh handle
    p.reset()
    assert np.array_equal(_bits(p.process(raw)), _bits(one))


def test_pfb_too_small_output_is_refused_without_state_change(sdr):
    import ctypes as C
    torch, dev = _torch()
    M, D = 32, 16
    h = gen.lowpass_taps(8 * M, 0.5 / M, 1.0)
    x = gen.complex_noise(10 * D + 5, 4)
    one = sdr.Pfb(h, M, D, "c64").process(x)
    p = sdr.Pfb(h, M, D, "c64")
    first = p.process(x[:D + 3])
    out = np.empty((one.shape[0], M), np.complex64)
    got = C.c_size_t(0)
    n_rest = x.size - (D + 3)
    need = p.output_count(n_rest)
    rest = np.ascontiguousarray(x[D + 3:])
    rc = sdr.lib().sdr_pfb_process(p.h, rest.ctypes.data, n_rest, out.ctypes.data, need - 1, M, C.byref(got))
    assert rc == 104 and got.value == 0
    d_in = torch.from_numpy(rest).to(dev)
    d_out = torch.empty((need, M), dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_pfb_process_dev(p.h, d_in.data_ptr(), n_rest, d_out.data_ptr(), need - 1, M, C.byref(got))
    assert rc == 104 and got.value == 0
    assert p.output_count(n_rest) == need
    second = p.process(rest)
    assert np.array_equal(_bits(np.concatenate([first, second])), _bits(one))


@pytest.mark.parametrize("M,D,L", [(64, 64, 16 * 64), (64, 32, 16 * 64 - 5), (64, 16, 8 * 64 - 1), (64, 8, 4 * 64),
                                   (1024, 1024, 32 * 1024), (8, 8, 13), (4096, 4096, 16 * 4096)])
@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_pfb_both_front_ends_agree_bit_for_bit(sdr, M, D, L, fmt):
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    n = max(40 * D, 3 * L) + 11
    raw, _ = _input(fmt, n, 12)
    a = sdr.Pfb(h, M, D, fmt).process(raw)
    b = sdr.Pfb(h, M, D, fmt, general=True).process(raw)
    assert a.shape == b.shape == (n // D, M)
    assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.parametrize("M,D,fmt", [(256, 128, "c64"), (64, 33, "u8iq"), (256, 128, "u8iq")])
def test_pfb_shards_concatenate_to_one_stream(sdr, M, D, fmt):
    torch, dev = _torch()
    from sdr_b200 import shard
    n = 1 << 22
    L = 16 * M
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    raw, _ = _input(fmt, n, 17)
    per = 2 if fmt == "u8iq" else 1
    es = 2 if fmt == "u8iq" else 8
    st = torch.cuda.current_stream(dev)
    d_raw = torch.from_numpy(np.ascontiguousarray(raw)).to(dev)
    base = d_raw.data_ptr()
    nf = n // D
    d_one = torch.empty((nf, M), dtype=torch.complex64, device=dev)
    assert sdr.Pfb(h, M, D, fmt, stream=st).process_dev(d_raw, n, d_one, nf) == nf
    torch.cuda.synchronize()
    one = d_one.cpu().numpy()
    halo = -(-(L - 1) // D) * D
    misaligned = 0
    for world in (2, 3):
        parts = []
        for rank in range(world):
            lo, hi, hlo = shard.sample_range(n, world, rank, halo=halo, align=D)
            p = sdr.Pfb(h, M, D, fmt, stream=st)
            cnt = p.output_count(hi - hlo)
            d_out = torch.empty((max(cnt, 1), M), dtype=torch.complex64, device=dev)
            misaligned += (base + hlo * es) % 16 != 0
            got = p.process_dev(base + hlo * es, hi - hlo, d_out, cnt)
            torch.cuda.synchronize()
            parts.append(d_out.cpu().numpy()[(lo - hlo) // D:got])
        cat = np.concatenate(parts)
        assert cat.shape == one.shape
        assert np.array_equal(_bits(cat), _bits(one))
    if fmt == "u8iq" and D % 2:
        assert misaligned > 0


@pytest.mark.parametrize("M,D,L,general", [(16, 5, 67, False), (16, 16, 53, False), (16, 16, 53, True),
                                           (64, 32, 16 * 64 - 7, False)])
def test_pfb_nan_poisons_exactly_its_windows(sdr, M, D, L, general):
    h = gen.lowpass_taps(L, 0.5 / M, 1.0)
    n = 20 * L
    x = gen.complex_noise(n, 2)
    s = n // 2 + 3
    x[s] = np.complex64(complex(np.nan, 0.0))
    y = sdr.Pfb(h, M, D, "c64", general=general).process(x)
    e = (np.arange(y.shape[0]) + 1) * D - 1
    hit = (e >= s) & (e - L + 1 <= s)
    assert hit.sum() >= 1
    assert np.isnan(y[hit]).all(axis=1).all()
    assert np.isfinite(y[~hit]).all()


def test_pfb_channel_major_feeds_pll_batch(sdr):
    torch, dev = _torch()
    M, D = 16, 8
    rate = 1.8e6
    h = gen.lowpass_taps(8 * M, 0.5 / M, 1.0)
    n = 4096 * D
    raw = gen.tone_noise_u8(n, rate, 3 * rate / M + 2e3, 0.5, 0.05, 5)
    frames = sdr.Pfb(h, M, D, "u8iq").process(raw)
    nf = frames.shape[0]
    design = sdr.PllDesign(0.0, 0.035, sdr.BiquadD.LowPass(8e3, .7), sdr.Identity(), sdr.Identity())
    want_v, want_l = sdr.PllBatch([design], M, rate / D).process(np.ascontiguousarray(frames.T))
    st = torch.cuda.current_stream(dev)
    stride = nf + 3
    d_in = torch.from_numpy(raw).to(dev)
    d_y = torch.empty((M, stride), dtype=torch.complex64, device=dev)
    assert sdr.Pfb(h, M, D, "u8iq", channel_major=True, stream=st).process_dev(d_in, n, d_y, nf, stride) == nf
    d_v = torch.empty((M, nf), dtype=torch.float32, device=dev)
    d_l = torch.empty((M, nf), dtype=torch.uint8, device=dev)
    sdr.PllBatch([design], M, rate / D, stream=st).process_dev(d_y, nf, d_v, d_l, in_stride=stride, out_stride=nf)
    torch.cuda.synchronize()
    assert np.array_equal(_bits(d_v.cpu().numpy()), _bits(want_v))
    assert np.array_equal(d_l.cpu().numpy(), want_l)


def test_pfb_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "pfb_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "PFB MIRROR OK" in r.stdout, r.stdout + r.stderr

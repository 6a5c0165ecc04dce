"""Polyphase synthesis filter bank (sdr_pfs): against the crate's own composition -- zero-stuff, Fir(f e^{+2 pi i k n / M})
per channel and a sum, through the CPU oracle -- and against f64 truth; the Pfb -> Pfs round trip; layout flags,
streaming, sharding, NaN bounds, draining and both back-end kernels."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import gen
import oracle_lib as O
import pfb_ref
import pfs_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = [(False, False), (True, False), (False, True), (True, True)]  # (shift, channel_major)


def _bar(M, x64):
    """the FFT bar of DESIGN.md section 4: 1e-5 log2(M) of max|x|"""
    return 1e-5 * max(1.0, np.log2(M)) * np.abs(x64).max()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _frames(n, M, seed):
    return gen.complex_noise(n * M, seed).reshape(n, M)


def _layout(y, shift, cmajor):
    """plain frames [n, M] in the layout Pfb writes with the same flags"""
    M = y.shape[1]
    if shift:
        y = y[:, (np.arange(M) - M // 2) % M]
    return np.ascontiguousarray(y.T if cmajor else y)


def _taps(L, M, D):
    """synthesis prototype: cutoff 1/M, gain D (Hamming; the Kaiser pair of pfs_ref is for round trips)"""
    return D * gen.lowpass_taps(L, 1.0 / M, 1.0) if L > 1 else np.array([0.5 * D], np.float32)


def _odd(M):
    return 5 if M <= 64 else (M // 3) | 1


@pytest.mark.parametrize("M", [8, 16])
@pytest.mark.parametrize("Dsel", ["M", "M/2", 3])
def test_pfs_pinned_to_stuff_fir_sum(sdr, M, Dsel):
    D = {"M": M, "M/2": M // 2}.get(Dsel, Dsel)
    L = 6 * M + 5
    f = gen.lowpass_taps(L, 1.0 / M, 1.0)
    y = _frames(300, M, 40 + M + D)
    got = sdr.Pfs(f, M, D).process(y)
    truth = R.direct_f64(f.astype(np.float64), y, M, D)
    oracle = R.direct_oracle_f32(f, y, M, D)
    assert got.shape == truth.shape == oracle.shape == (300 * D,)
    bar = _bar(M, truth)
    assert np.abs(got - truth).max() <= bar
    assert np.abs(got - oracle).max() <= bar


@pytest.mark.parametrize("shift,cmajor", LAYOUTS)
@pytest.mark.parametrize("M", [8, 16, 64, 1024, 4096, 1000])
@pytest.mark.parametrize("Dsel", ["M", "M/2", "odd"])
def test_pfs_against_f64(sdr, M, Dsel, shift, cmajor):
    D = {"M": M, "M/2": M // 2, "odd": _odd(M)}[Dsel]
    L = 12 * M + 1
    f = _taps(L, M, D)
    nf = max(64, (1 << 20) // D)
    y = _frames(nf, M, 7 + M + D)
    got = sdr.Pfs(f, M, D, shift=shift, channel_major=cmajor).process(_layout(y, shift, cmajor))
    assert got.shape == (nf * D,)
    n = nf * D
    pick = np.unique(np.concatenate([np.arange(min(n, 3000)), np.arange(n // 2, n // 2 + 1000), np.arange(n - 3000, n)]))
    truth = R.polyphase_f64(f, y, M, D, outputs=pick)
    assert np.abs(got[pick] - truth).max() <= _bar(M, truth)
    assert np.isfinite(got).all()


def test_pfs_spot_outputs_at_2_28(sdr):
    torch, dev = _torch()
    M, D = 1024, 512
    f = R.prototype_pair(M, D, 12)[1]
    nf = (1 << 28) // D
    g = torch.Generator(device=dev).manual_seed(5)
    d_y = torch.randn((nf, M), dtype=torch.complex64, device=dev, generator=g)
    d_out = torch.empty(nf * D, dtype=torch.complex64, device=dev)
    st = torch.cuda.current_stream(dev)
    assert sdr.Pfs(f, M, D, stream=st).process_dev(d_y, nf, d_out, nf * D) == nf * D
    torch.cuda.synchronize()
    n = nf * D
    for t0 in (0, n // 3 + 77, n - 4096):
        pick = np.arange(t0, t0 + 4096)
        f0 = max(0, t0 // D - 30)
        y = d_y[f0:(t0 + 4096) // D + 1].cpu().numpy()  # every frame the picked outputs reach
        truth = R.polyphase_f64(f, y, M, D, outputs=pick - f0 * D)
        got = d_out[t0:t0 + 4096].cpu().numpy()
        assert np.abs(got - truth).max() <= _bar(M, truth), t0
    del d_y, d_out


@pytest.mark.parametrize("M,D,L", [(16, 5, 8 * 16 + 3), (1024, 512, 12 * 1024 + 1), (1000, 1000, 16001),
                                   (64, 16, 8 * 64 - 1)])
def test_pfs_layouts_and_strides_are_exact(sdr, M, D, L):
    torch, dev = _torch()
    f = _taps(L, M, D)
    nf = 3 * (-(-L // D)) + 37
    y = _frames(nf, M, 3)
    plain = sdr.Pfs(f, M, D).process(y)
    st = torch.cuda.current_stream(dev)
    for shift, cmajor in LAYOUTS:
        host = sdr.Pfs(f, M, D, shift=shift, channel_major=cmajor).process(_layout(y, shift, cmajor))
        assert np.array_equal(_bits(host), _bits(plain)), (shift, cmajor)
        # device entry point with an odd stride: frames of M + 3, or M rows of nf + 5
        lay = _layout(y, shift, cmajor)
        pad = np.full((M, nf + 5) if cmajor else (nf, M + 3), np.nan, np.complex64)
        pad[:, :lay.shape[1]] = lay
        d_in = torch.from_numpy(pad).to(dev)
        d_out = torch.full((nf * D + 7,), float("nan"), dtype=torch.complex64, device=dev)
        p = sdr.Pfs(f, M, D, shift=shift, channel_major=cmajor, stream=st)
        assert p.process_dev(d_in, nf, d_out, nf * D + 7, pad.shape[1]) == nf * D
        torch.cuda.synchronize()
        out = d_out.cpu().numpy()
        assert np.array_equal(_bits(out[:nf * D]), _bits(plain)) and np.isnan(out[nf * D:]).all(), (shift, cmajor)


@pytest.mark.parametrize("M,D,L", [(64, 64, 12 * 64 + 1), (64, 32, 12 * 64 + 1), (64, 16, 4 * 64 - 3), (64, 8, 2 * 64),
                                   (1024, 1024, 30 * 1024), (1024, 512, 12 * 1024 + 1), (8, 8, 13), (16, 16, 1),
                                   (4096, 2048, 12 * 4096 + 1)])
def test_pfs_both_back_ends_agree_bit_for_bit(sdr, M, D, L):
    f = _taps(L, M, D)
    nf = 2 * (-(-L // D)) + 300
    y = _frames(nf, M, 12)
    a = sdr.Pfs(f, M, D).process(y)
    b = sdr.Pfs(f, M, D, general=True).process(y)
    assert a.shape == b.shape == (nf * D,)
    assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.parametrize("M,D,L,general", [(64, 32, 12 * 64 + 1, False), (64, 32, 12 * 64 + 1, True),
                                           (16, 5, 67, False), (1000, 500, 4001, False)])
def test_pfs_streaming_clone_reset(sdr, M, D, L, general):
    f = _taps(L, M, D)
    nf = 200
    y = _frames(nf, M, 9)
    one = sdr.Pfs(f, M, D, general=general).process(y)
    # one frame per call
    p = sdr.Pfs(f, M, D, general=general)
    parts = [p.process(y[m:m + 1]) for m in range(nf)]
    assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
    # random blockings, a clone mid-stream
    rng = np.random.default_rng(M + D)
    for _ in range(2):
        p = sdr.Pfs(f, M, D, general=general)
        parts, pos, clone = [], 0, None
        while pos < nf:
            b = int(min(nf - pos, rng.integers(0, 40)))
            parts.append(p.process(y[pos:pos + b]))
            pos += b
            if clone is None and pos > nf // 2:
                clone, at = p.clone(), pos
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
        assert np.array_equal(_bits(clone.process(y[at:])), _bits(one[at * D:]))
    p.reset()
    assert np.array_equal(_bits(p.process(y)), _bits(one))


def test_pfs_too_small_output_is_refused_without_state_change(sdr):
    torch, dev = _torch()
    M, D = 32, 16
    f = _taps(8 * M + 1, M, D)
    y = _frames(40, M, 4)
    one = sdr.Pfs(f, M, D).process(y)
    p = sdr.Pfs(f, M, D)
    first = p.process(y[:7])
    rest = np.ascontiguousarray(y[7:])
    need = p.output_count(rest.shape[0])
    assert need == rest.shape[0] * D
    out = np.empty(need, np.complex64)
    got = C.c_size_t(0)
    rc = sdr.lib().sdr_pfs_process(p.h, rest.ctypes.data, rest.shape[0], M, out.ctypes.data, need - 1, C.byref(got))
    assert rc == 104 and got.value == 0
    d_in = torch.from_numpy(rest).to(dev)
    d_out = torch.empty(need, dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_pfs_process_dev(p.h, d_in.data_ptr(), rest.shape[0], M, d_out.data_ptr(), need - 1,
                                       C.byref(got))
    assert rc == 104 and got.value == 0
    second = p.process(rest)
    assert np.array_equal(_bits(np.concatenate([first, second])), _bits(one))


@pytest.mark.parametrize("M,D,L", [(256, 128, 12 * 256 + 1), (64, 5, 300), (1024, 1024, 16 * 1024)])
def test_pfs_shards_concatenate_to_one_stream(sdr, M, D, L):
    """a shard starting at frame f0, primed with the H = ceil((L - 1) / D) frames before it and with its first H D
    outputs dropped, gives the bits of one stream"""
    torch, dev = _torch()
    f = _taps(L, M, D)
    nf = 3000
    H = -(-(L - 1) // D)
    st = torch.cuda.current_stream(dev)
    d_y = torch.from_numpy(_frames(nf, M, 17)).to(dev)
    d_one = torch.empty(nf * D, dtype=torch.complex64, device=dev)
    sdr.Pfs(f, M, D, stream=st).process_dev(d_y, nf, d_one, nf * D)
    torch.cuda.synchronize()
    one = d_one.cpu().numpy()
    for world in (2, 3):
        cuts = [nf * r // world for r in range(world + 1)]
        parts = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            plo = max(0, lo - H)
            d_out = torch.empty((hi - plo) * D, dtype=torch.complex64, device=dev)
            sdr.Pfs(f, M, D, stream=st).process_dev(d_y[plo:hi], hi - plo, d_out, (hi - plo) * D)
            torch.cuda.synchronize()
            parts.append(d_out.cpu().numpy()[(lo - plo) * D:])
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))


@pytest.mark.parametrize("M,D,L,general", [(16, 5, 67, False), (16, 16, 53, False), (16, 16, 53, True),
                                           (64, 32, 12 * 64 + 1, False), (64, 32, 12 * 64 + 1, True)])
def test_pfs_nan_poisons_exactly_its_outputs(sdr, M, D, L, general):
    f = _taps(L, M, D)
    f[L // 2] = 0.0  # a zero tap is still multiplied
    nf = 4 * (-(-L // D)) + 20
    y = _frames(nf, M, 2)
    m = nf // 2
    y[m, 3] = np.complex64(complex(np.nan, 0.0))
    x = sdr.Pfs(f, M, D, general=general).process(y)
    t = np.arange(x.size)
    hit = (t >= (m + 1) * D - 1) & (t < (m + 1) * D - 1 + L)
    assert np.isnan(x[hit]).all()
    assert np.isfinite(x[~hit]).all()


@pytest.mark.parametrize("M,D,L", [(16, 8, 12 * 16 + 1), (16, 5, 67), (8, 8, 1)])
def test_pfs_zero_frames_drain_the_tail(sdr, M, D, L):
    f = _taps(L, M, D)
    H = -(-(L - 1) // D)
    nf = 50
    y = _frames(nf, M, 8)
    p = sdr.Pfs(f, M, D)
    body = p.process(y)
    tail = p.process(np.zeros((H, M), np.complex64)) if H else np.zeros(0, np.complex64)
    got = np.concatenate([body, tail])
    # the whole linear convolution of every zero-stuffed channel: nf D + L - 1 samples, the last nonzero at nf D + L - 2
    full = np.zeros(nf * D + L - 1, np.complex128)
    for k in range(M):
        full += np.convolve(R.zero_stuff(y[:, k].astype(np.complex128), D), R.modulated_taps(f, M, k))
    assert got.size == (nf + H) * D >= full.size
    full = np.concatenate([full, np.zeros(got.size - full.size)])
    assert np.abs(got - full).max() <= _bar(M, full)
    assert np.abs(p.process(np.zeros((3, M), np.complex64))).max() == 0


@pytest.mark.parametrize("M,D,T,k0", [(16, 8, 12, 3), (64, 32, 12, 45), (1024, 512, 12, 300)])
def test_pfs_known_answer_single_channel(sdr, M, D, T, k0):
    """channel k0 alone holding e^{2 pi i k0 ((m+1) D - 1) / M}, the rotation sdr_pfb leaves on a channel's DC content,
    synthesises e^{2 pi i k0 t / M} after the first L samples, in every layout"""
    f = R.prototype_pair(M, D, T)[1]
    L = f.size
    nf = max(600, 4 * L // D)
    m = np.arange(nf)
    y = np.zeros((nf, M), np.complex64)
    y[:, k0] = np.exp(2j * np.pi * k0 * (((m + 1) * D - 1) % M) / M)
    t = np.arange(nf * D)
    tone = np.exp(2j * np.pi * k0 * (t % M) / M)
    pick = t[L:]
    x64 = R.polyphase_f64(f, y, M, D, outputs=pick)
    err64 = np.abs(x64 - tone[pick]).max()  # the filter's own error, not round-off
    for shift, cmajor in LAYOUTS:
        x = sdr.Pfs(f, M, D, shift=shift, channel_major=cmajor).process(_layout(y, shift, cmajor))
        assert np.abs(x[L:] - tone[L:]).max() <= err64 + _bar(M, tone), (shift, cmajor)


def _cascade_bar(M, D, f, y64, x64):
    """f32 analysis -> f32 synthesis against the f64 cascade: the analysis bar eps_a per channel sample, carried
    through synthesis as errors incoherent across channels and taps (RMS sqrt(M sum_{n = c (D)} f[n]^2) eps_a), plus
    the synthesis bar"""
    eps_a = _bar(M, y64)
    f = np.asarray(f, np.float64)
    ff = max((f[c::D] ** 2).sum() for c in range(D))
    return eps_a * np.sqrt(M * ff) + _bar(M, x64)


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_pfb_pfs_round_trip(sdr, fmt):
    torch, dev = _torch()
    M, D, T = 1024, 512, 12
    h, f = R.prototype_pair(M, D, T)
    n = 1 << 21
    if fmt == "u8iq":
        raw = gen.random_u8(2 * n, 31)
        x = O.unpack_u8iq(raw)
    else:
        raw = x = gen.complex_noise(n, 31)
    nf = n // D
    # host path
    frames = sdr.Pfb(h, M, D, fmt).process(raw)
    host = sdr.Pfs(f, M, D).process(frames)
    assert host.shape == (n,)
    # device path: the pfb output buffer goes straight in, frame-major and channel-major
    st = torch.cuda.current_stream(dev)
    d_in = torch.from_numpy(np.ascontiguousarray(raw)).to(dev)
    for cmajor in (False, True):
        d_y = torch.empty((M, nf) if cmajor else (nf, M), dtype=torch.complex64, device=dev)
        assert sdr.Pfb(h, M, D, fmt, channel_major=cmajor, stream=st).process_dev(d_in, n, d_y, nf) == nf
        d_x = torch.empty(n, dtype=torch.complex64, device=dev)
        assert sdr.Pfs(f, M, D, channel_major=cmajor, stream=st).process_dev(d_y, nf, d_x, n) == n
        torch.cuda.synchronize()
        assert np.array_equal(_bits(d_x.cpu().numpy()), _bits(host)), cmajor
    # against the f64 cascade and against the delayed input, on spot stretches past the start-up transient
    d = T * M
    starts = (4 * d, n - 8192)
    pick = np.concatenate([np.arange(a, a + 8192) for a in starts])
    need = np.unique(np.concatenate([np.arange(a // D - 2 * T - 2, (a + 8192) // D) for a in starts]))
    y64 = np.zeros((nf, M), np.complex128)
    y64[need] = pfb_ref.polyphase_f64(h, x, M, D, frames=need)
    x64 = R.polyphase_f64(f, y64, M, D, outputs=pick)
    bar = _cascade_bar(M, D, f, y64[need], x64)
    assert np.abs(host[pick] - x64).max() <= bar
    own = np.abs(x64 - x[pick - d]).max()
    assert np.abs(host[pick] - x[pick - d]).max() <= own + bar
    ref = x[pick - d].astype(np.complex128)
    snr = 10 * np.log10(np.mean(np.abs(ref) ** 2) / np.mean(np.abs(host[pick] - ref) ** 2))
    print("pfb -> pfs round trip (%s, M=%d D=%d T=%d): %.1f dB SNR, f64 cascade %.1f dB" % (
        fmt, M, D, T, snr, 10 * np.log10(np.mean(np.abs(ref) ** 2) / np.mean(np.abs(x64 - ref) ** 2))))


def test_pfs_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "pfs_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "PFS MIRROR OK" in r.stdout, r.stdout + r.stderr

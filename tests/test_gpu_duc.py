"""Digital up-converter bank (sdr_duc): against f64 truth with exact integer phases and against the crate's own
composition (zero-stuff, Fir(h_k), an f32 mix, the sum) through the CPU oracle; a known answer; agreement with sdr_pfs
on the channel grid; the adjoint identity and the round trip with GPU sdr_ddc; streaming, clones, shards, NaN bounds
and draining."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ddc_ref
import duc_ref as R
import gen
import oracle_lib as O
import pfs_ref
from test_duc_host import F_BIG, F_TOP, ROUND_TRIP_SNR_DB, round_trip_input

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TWO64 = 1 << 64


def _bar(x64):
    return 1e-5 * np.abs(x64).max()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _freqs(C_, seed):
    return np.random.default_rng(seed).uniform(-0.5, 0.5, C_)


def _taps(C_, L, I, shared, seed=0):
    """low-pass taps (cutoff 0.5/I, gain I), one row per channel (slightly different cutoffs) unless shared"""
    if L == 1:
        t = np.full((1 if shared else C_, 1), float(I), np.float32)
    else:
        t = np.stack([I * gen.lowpass_taps(L, (0.45 + 0.05 * k / max(C_, 1)) / I, 1.0)
                      for k in range(1 if shared else C_)])
    return t[0] if shared else t


def _rows(C_, n, seed):
    return gen.complex_noise(C_ * n, seed).reshape(C_, n)


def _incs(bank):
    return [int(v) for v in bank.phase_inc]


@pytest.mark.parametrize("C_,I,L,shared", [
    (1, 1, 1, True), (1, 8, 255, True), (3, 2, 64, False), (3, 10, 1000, True), (8, 8, 255, False),
    (8, 32, 511, True), (17, 10, 64, False), (17, 1, 255, True), (256, 8, 64, True), (256, 2, 255, False),
    (8, 1, 1000, False), (3, 32, 1, False)])
def test_duc_against_f64_and_oracle(sdr, C_, I, L, shared):
    h = _taps(C_, L, I, shared, C_)
    nf = max(64, min(20000 // I, 4000000 // (I * -(-L // I)))) if C_ < 256 else 200
    y = _rows(C_, nf, C_ + I + L)
    bank = sdr.Duc(h, _freqs(C_, C_ + L), 1.0, I, first_sample=F_BIG)
    got = bank.process(y)
    assert got.shape == (nf * I,)
    incs = _incs(bank)
    truth = R.computed_f64(h.astype(np.float64), y, incs, I, F_BIG)
    assert np.abs(got - truth).max() <= _bar(truth)
    if C_ <= 17:
        oracle = R.oracle_f32(h, y, incs, I, F_BIG)
        assert np.abs(got - oracle).max() <= _bar(truth)


@pytest.mark.parametrize("F", [0, F_BIG, F_TOP])
def test_duc_stream_position_against_f64(sdr, F):
    C_, I, L = 3, 8, 255
    h = _taps(C_, L, I, False)
    y = _rows(C_, 3000, 5)
    bank = sdr.Duc(h, _freqs(C_, 9), 1.0, I, first_sample=F)
    got = bank.process(y)
    truth = R.computed_f64(h.astype(np.float64), y, _incs(bank), I, F)
    assert np.abs(got - truth).max() <= _bar(truth)


@pytest.mark.parametrize("I,L", [(8, 255), (10, 1000), (1, 64), (32, 511)])
def test_duc_known_answer_constant_channel(sdr, I, L):
    """a constant a in channel k alone gives a S_{(n+1) mod I} e^{+2 pi i phi_k(F + n)} after L - 1 samples"""
    C_, k, a = 4, 2, np.complex64(0.75 - 0.5j)
    h = _taps(C_, L, I, False)
    nf = 4 * L // I + 200
    y = np.zeros((C_, nf), np.complex64)
    y[k] = a
    bank = sdr.Duc(h, _freqs(C_, 3), 1.0, I, first_sample=F_TOP)
    x = bank.process(y)
    n = np.arange(L - 1, nf * I)
    S = np.array([h[k][c::I].astype(np.float64).sum() for c in range(I)])
    want = a * S[(n + 1) % I] * R.rot_up(ddc_ref.phases(F_TOP, n, _incs(bank)[k]))
    assert np.abs(x[L - 1:] - want).max() <= 1e-5 * np.abs(want).max()


@pytest.mark.parametrize("M", [8, 16, 64])
def test_duc_on_the_channel_grid_equals_pfs(sdr, M):
    """Delta_k = k 2^64 / M, shared taps, I = D: the bank equals sdr_pfs fed y_k[m] e^{+2 pi i k (F + (m+1) D - 1) / M}"""
    D, L, F = M // 2, 12 * M + 1, 12345
    f = pfs_ref.prototype_pair(M, D, 12)[1].astype(np.float32)
    nf = 2000
    y = _rows(M, nf, M)
    bank = sdr.Duc(f, np.arange(M) / M, 1.0, D, first_sample=F)
    assert _incs(bank) == [(k * TWO64 // M) % TWO64 for k in range(M)]
    x = bank.process(y)
    m = np.arange(nf)
    tw = np.exp(2j * np.pi * np.outer(np.arange(M), (F + (m + 1) * D - 1) % M) / M)
    frames = (y * tw).astype(np.complex64).T
    xp = sdr.Pfs(f, M, D).process(frames)
    truth = R.computed_f64(f.astype(np.float64), y, _incs(bank), D, F)
    bar = _bar(truth) + 1e-5 * np.log2(M) * np.abs(truth).max()
    assert np.abs(x - xp).max() <= bar


def test_duc_adjoint_of_gpu_ddc(sdr):
    C_, D, L, F = 3, 5, 23, F_BIG
    rng = np.random.default_rng(4)
    h = rng.standard_normal((C_, L)).astype(np.float32)
    freqs = _freqs(C_, 4)
    nf = 4000
    x = gen.complex_noise(nf * D, 6)
    v = _rows(C_, nf, 7)
    H = -(-(L - 1) // D)
    yd = sdr.Ddc(h, freqs, 1.0, D, "c64", first_sample=F).process(x)
    xh = sdr.Duc(np.ascontiguousarray(h[:, ::-1]), freqs, 1.0, D, first_sample=(F - (L - 1)) % TWO64).process(
        np.concatenate([v, np.zeros((C_, H), np.complex64)], axis=1))
    lhs = np.sum(np.conj(v.astype(np.complex128)) * yd)
    rhs = np.sum(np.conj(xh[L - 1:L - 1 + nf * D].astype(np.complex128)) * x)
    # each side is a sum of C nf (resp. nf D) terms with relative error <~ 1e-5 of the largest: bound incoherently
    scale = np.sqrt(np.sum(np.abs(v) ** 2) * np.sum(np.abs(yd) ** 2)) + np.sqrt(
        np.sum(np.abs(xh) ** 2) * np.sum(np.abs(x) ** 2))
    assert abs(lhs - rhs) <= 1e-5 * scale


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_ddc_duc_round_trip(sdr, fmt):
    torch, dev = _torch()
    D, T = 8, 64
    h, f = R.kaiser_pair(D, T)
    h, f = h.astype(np.float32), f.astype(np.float32)
    nus = (-0.3, 0.05, 0.27)
    n, F = 1 << 15, F_BIG  # the host round trip's input and its f64 figure
    if fmt == "u8iq":
        raw = gen.random_u8(2 * n, 31)
        x = O.unpack_u8iq(raw).astype(np.complex128)
        incs = [ddc_ref.phase_increment_exact(nu, 1.0) for nu in nus]
    else:
        x, incs = round_trip_input(n, F, nus)
        raw = x.astype(np.complex64)
    d = T * D
    nf = n // D
    ddc = sdr.Ddc(h, nus, 1.0, D, fmt, first_sample=F)
    y = ddc.process(raw)
    host = sdr.Duc(f, nus, 1.0, D, first_sample=(F - d) % TWO64).process(y)
    assert host.shape == (n,)
    # device path with sdr_ddc's output rows at its out_stride
    st = torch.cuda.current_stream(dev)
    stride = nf + 7
    d_in = torch.from_numpy(np.ascontiguousarray(raw)).to(dev)
    d_y = torch.zeros((len(nus), stride), dtype=torch.complex64, device=dev)
    assert sdr.Ddc(h, nus, 1.0, D, fmt, first_sample=F, stream=st).process_dev(d_in, n, d_y, nf, stride) == nf
    d_x = torch.empty(n, dtype=torch.complex64, device=dev)
    assert sdr.Duc(f, nus, 1.0, D, first_sample=(F - d) % TWO64, stream=st).process_dev(d_y, nf, d_x, n, stride) == n
    torch.cuda.synchronize()
    assert np.array_equal(_bits(d_x.cpu().numpy()), _bits(host))
    # against the f64 cascade (ddc bar carried through the synthesis taps, plus the duc bar)
    y64 = ddc_ref.mix_first_f64(h.astype(np.float64), x, incs, D, F)
    x64 = R.computed_f64(f.astype(np.float64), y64, incs, D, (F - d) % TWO64)
    ff = max(np.sqrt((f[c::D].astype(np.float64) ** 2).sum()) for c in range(D))
    bar = 1e-5 * np.abs(y64).max() * ff * np.sqrt(len(nus)) + _bar(x64)
    assert np.abs(host - x64).max() <= bar
    if fmt == "c64":
        ref = x[3 * d:n - d]
        sig = np.mean(np.abs(ref) ** 2)
        snr = 10 * np.log10(sig / np.mean(np.abs(host[4 * d:] - ref) ** 2))
        snr64 = 10 * np.log10(sig / np.mean(np.abs(x64[4 * d:] - ref) ** 2))
        print("ddc -> duc round trip: %.1f dB (f64 cascade %.1f dB)" % (snr, snr64))
        assert snr64 >= ROUND_TRIP_SNR_DB and snr >= snr64 - 1, (snr, snr64)


@pytest.mark.parametrize("C_,I,L", [(3, 8, 255), (5, 10, 64), (2, 1, 100), (4, 200, 1000), (1, 3, 1)])
def test_duc_streaming_clone_reset_retry(sdr, C_, I, L):
    h = _taps(C_, L, I, False)
    freqs = _freqs(C_, 2)
    nf = 300
    y = _rows(C_, nf, 9)
    one = sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG).process(y)
    p = sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG)
    parts = [p.process(y[:, m:m + 1]) for m in range(nf)]
    assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
    rng = np.random.default_rng(C_ + I)
    for _ in range(2):
        p = sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG)
        parts, pos, clone = [], 0, None
        while pos < nf:
            b = int(min(nf - pos, rng.integers(0, 50)))
            parts.append(p.process(y[:, pos:pos + b]))
            pos += b
            if clone is None and pos > nf // 2:
                clone, at = p.clone(), pos
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
        assert np.array_equal(_bits(clone.process(y[:, at:])), _bits(one[at * I:]))
    p.reset()
    assert np.array_equal(_bits(p.process(y)), _bits(one))
    # a too-small output is refused before any state changes, host and device
    torch, dev = _torch()
    p = sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG)
    first = p.process(y[:, :7])
    rest = np.ascontiguousarray(y[:, 7:])
    need = p.output_count(rest.shape[1])
    assert need == rest.shape[1] * I
    out = np.empty(need, np.complex64)
    got = C.c_size_t(0)
    rc = sdr.lib().sdr_duc_process(p.h, rest.ctypes.data, rest.shape[1], rest.shape[1], out.ctypes.data, need - 1,
                                   C.byref(got))
    assert rc == 104 and got.value == 0
    d_in = torch.from_numpy(rest).to(dev)
    d_out = torch.empty(need, dtype=torch.complex64, device=dev)
    rc = sdr.lib().sdr_duc_process_dev(p.h, d_in.data_ptr(), rest.shape[1], rest.shape[1], d_out.data_ptr(), need - 1,
                                       C.byref(got))
    assert rc == 104 and got.value == 0
    assert np.array_equal(_bits(np.concatenate([first, p.process(rest)])), _bits(one))


@pytest.mark.parametrize("C_,I,L", [(3, 8, 255), (4, 5, 300), (2, 64, 4095)])
def test_duc_odd_strides_and_shards(sdr, C_, I, L):
    """odd device row strides give the host bits; a shard primed with the H frames before it, with first_sample the
    primed frame's absolute output index and its first H I outputs dropped, gives one stream's bits"""
    torch, dev = _torch()
    h = _taps(C_, L, I, True)
    freqs = _freqs(C_, 8)
    nf = 1500
    y = _rows(C_, nf, 17)
    one = sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG).process(y)
    st = torch.cuda.current_stream(dev)
    pad = np.full((C_, nf + 5), np.nan, np.complex64)
    pad[:, :nf] = y
    d_y = torch.from_numpy(pad).to(dev)
    d_out = torch.full((nf * I + 3,), float("nan"), dtype=torch.complex64, device=dev)
    assert sdr.Duc(h, freqs, 1.0, I, first_sample=F_BIG, stream=st).process_dev(d_y, nf, d_out, nf * I + 3,
                                                                               nf + 5) == nf * I
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    assert np.array_equal(_bits(out[:nf * I]), _bits(one)) and np.isnan(out[nf * I:]).all()
    H = -(-(L - 1) // I)
    for world in (2, 3):
        cuts = [nf * r // world for r in range(world + 1)]
        parts = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            plo = max(0, lo - H)
            b = sdr.Duc(h, freqs, 1.0, I, first_sample=(F_BIG + plo * I) % TWO64)
            parts.append(b.process(y[:, plo:hi])[(lo - plo) * I:])
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))


@pytest.mark.parametrize("I,L", [(8, 255), (5, 67), (1, 16), (200, 1000)])
def test_duc_nan_poisons_exactly_its_outputs_and_zero_frames_drain(sdr, I, L):
    C_ = 3
    h = _taps(C_, L, I, False)
    h[1][L // 2] = 0.0  # a zero tap is still multiplied
    freqs = _freqs(C_, 1)
    nf = 4 * (-(-L // I)) + 20
    y = _rows(C_, nf, 2)
    m = nf // 2
    y[1, m] = np.complex64(complex(np.nan, 0.0))
    clean = y.copy()
    clean[1, m] = 0
    x = sdr.Duc(h, freqs, 1.0, I).process(y)
    ref = sdr.Duc(h, freqs, 1.0, I).process(clean)
    t = np.arange(x.size)
    hit = (t >= (m + 1) * I - 1) & (t < (m + 1) * I - 1 + L)
    assert np.isnan(x[hit]).all()
    assert np.array_equal(_bits(x[~hit]), _bits(ref[~hit]))
    # drain: ceil((L - 1) / I) zero frames bring out the whole tail
    H = -(-(L - 1) // I)
    p = sdr.Duc(h, freqs, 1.0, I)
    got = np.concatenate([p.process(clean), p.process(np.zeros((C_, H), np.complex64))])
    full = R.definition_f64(h.astype(np.float64), np.concatenate([clean, np.zeros((C_, H))], axis=1), _incs(p), I)
    assert got.size == full.size >= nf * I + L - 1
    assert np.abs(got - full).max() <= _bar(full)
    assert np.abs(p.process(np.zeros((C_, 3), np.complex64))).max() == 0


def test_duc_spot_outputs_at_2_28(sdr):
    torch, dev = _torch()
    C_, I, L = 8, 8, 255
    h = _taps(C_, L, I, False)
    nf = (1 << 28) // I
    g = torch.Generator(device=dev).manual_seed(5)
    d_y = torch.randn((C_, nf), dtype=torch.complex64, device=dev, generator=g)
    d_out = torch.empty(nf * I, dtype=torch.complex64, device=dev)
    st = torch.cuda.current_stream(dev)
    bank = sdr.Duc(h, _freqs(C_, 11), 1.0, I, first_sample=F_BIG, stream=st)
    assert bank.process_dev(d_y, nf, d_out, nf * I) == nf * I
    torch.cuda.synchronize()
    n = nf * I
    for t0 in (0, n // 3 + 77, n - 4096):
        f0 = max(0, t0 // I - L // I - 2)
        y = d_y[:, f0:(t0 + 4096) // I + 1].cpu().numpy()
        truth = R.computed_f64(h.astype(np.float64), y, _incs(bank), I, (F_BIG + f0 * I) % TWO64,
                               outputs=np.arange(t0, t0 + 4096) - f0 * I)
        got = d_out[t0:t0 + 4096].cpu().numpy()
        assert np.abs(got - truth).max() <= _bar(truth), t0
    del d_y, d_out


def test_duc_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "duc_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DUC MIRROR OK" in r.stdout, r.stdout + r.stderr

"""GPU: averaged power spectra (sdr_psd).  Every spectrum against the f64 reference over a grid of N, hop and K on both
paths; the composition with WindowFft; known answers (a Hann-tapered tone, Parseval); a 2^28-sample run on the fused
path; NaN poisoning; bit-identity across blockings, clone, reset, the too-small retry, unaligned addresses and shards;
signal.power_spectra; the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import gen
import oracle_lib as O
import psd_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _input(fmt, n, seed):
    """(what the handle is fed, the same samples as complex128)"""
    if fmt == "u8iq":
        raw = gen.random_u8(2 * n, seed)
        return raw, O.unpack_u8iq(raw).astype(np.complex128)
    x = gen.complex_noise(n, seed)
    return x, x.astype(np.complex128)


def _check(got, want, N):
    assert got.shape == want.shape, (got.shape, want.shape)
    for g in range(want.shape[0]):
        mx = np.abs(want[g]).max()
        err = np.abs(got[g].astype(np.float64) - want[g]).max()
        assert err <= R.bar(N) * mx, (g, float(err), float(mx))


def _hops(N):
    return sorted({h for h in (N, N // 2, N // 4, 3, N + 17) if h >= 1})


GRID = [(N, H, K) for N in (1, 16, 256, 1000, 1024, 4096, 65536) for H in _hops(N) for K in (1, 3, 32, 33, 100)]


@pytest.mark.parametrize("N,H,K", GRID)
def test_psd_grid_against_f64(sdr, N, H, K):
    i = GRID.index((N, H, K))
    G = 2 if N * K * max(H, 1) > (1 << 24) else 3
    n = G * K * H + (i % 5) * 7 % (K * H)  # a few samples past the last complete spectrum
    # two variants per point, cycling the formats, tapers and flags over the grid
    variants = [("u8iq", True, (True, True)), ("c64", False, [(True, False), (False, True), (False, False)][i % 3])]
    if i % 2:
        variants = [("c64", True, (True, True)), ("u8iq", False, [(False, False), (True, False), (False, True)][i % 3])]
    for fmt, hann, (shift, norm) in variants:
        raw, x = _input(fmt, n, 100 + i)
        w = np.hanning(N).astype(np.float32) if hann and N > 1 else None
        p = sdr.Psd(N, H, K, window=w, fmt=fmt, shift=shift, norm=norm)
        assert p.output_count(n) == G
        got = p.process(raw)
        assert p.last_path == (2 if N == 1024 else 1)
        want = R.power_f64(x, N, H, K, None if w is None else w.astype(np.float64), shift, norm)
        _check(got, want, N)
        p.close()


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("general", [False, True])
@pytest.mark.parametrize("N,H", [(1024, 1024), (1024, 333), (1000, 250)])
def test_psd_equals_mean_of_window_fft_power(sdr, fmt, general, N, H):
    K, n = 7, 40000
    raw, _ = _input(fmt, n, 5)
    X = sdr.WindowFft(N, H, fmt).process(raw)
    G = X.shape[0] // K
    want = (np.abs(X[:G * K].astype(np.complex128)) ** 2).reshape(G, K, N).mean(axis=1)
    p = sdr.Psd(N, H, K, fmt=fmt, general=general)
    got = p.process(raw)
    assert p.last_path == (2 if N == 1024 and not general else 1)
    _check(got, want, N)


@pytest.mark.parametrize("N,general", [(1024, False), (1024, True), (1000, False)])
def test_hann_tone_known_answer(sdr, N, general):
    b, A, K = 37, 0.5, 4
    n = N * K * 3
    t = np.arange(n)
    x = (A * np.exp(2j * np.pi * b * t / N)).astype(np.complex64)
    w = np.hanning(N + 1)[:N]  # periodic Hann: the tone's energy lands on bins b - 1, b, b + 1 only
    p = sdr.Psd(N, N, K, window=w.astype(np.float32), fmt="c64", general=general)
    P = p.process(x)
    assert P.shape == (3, N)
    want = A * A * w.astype(np.float32).astype(np.float64).sum() ** 2 / N
    for g in range(1, 3):  # spectrum 0 starts inside the tone too: every frame is full
        assert int(np.argmax(P[g])) == b + N // 2
        assert abs(P[g][b + N // 2] - want) <= 1e-5 * want


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,H,K,general", [(1024, 512, 33, False), (1024, 3, 5, False), (1000, 400, 40, False),
                                           (1024, 1024, 2, True)])
def test_parseval_per_spectrum(sdr, fmt, N, H, K, general):
    n = 3 * K * H + 11
    raw, x = _input(fmt, n, 9)
    w = np.hanning(N).astype(np.float32)
    got = sdr.Psd(N, H, K, window=w, fmt=fmt, shift=True, norm=False, general=general).process(raw)
    fr = R.frames(x, N, H, got.shape[0] * K) * w.astype(np.float64)
    energy = (np.abs(fr) ** 2).sum(axis=1).reshape(-1, K).sum(axis=1)
    want = N / K * energy  # sum_k |X_k|^2 = N sum_n |x_n|^2 for each frame
    tot = got.astype(np.float64).sum(axis=1)
    assert np.abs(tot - want).max() <= R.bar(N) * want.max()


def test_product_size_on_the_fused_path(sdr):
    torch, dev = _torch()
    n, N, K = 1 << 28, 1024, 256
    G = n // N // K
    raw = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    p = sdr.Psd(N, N, K, fmt="u8iq", shift=True, norm=False, stream=st)
    out = torch.empty((G, N), dtype=torch.float32, device=dev)
    assert p.process_dev(raw, n, out, G) == G
    torch.cuda.synchronize()
    assert p.last_path == 2
    # Parseval on every spectrum, in f64 on the device
    x = (raw.view(-1, 2).to(torch.float64) - 128.0) / 128.0
    energy = (x * x).sum(dim=1).view(G, K * N).sum(dim=1)
    want = (N / K * energy).cpu().numpy()
    tot = out.to(torch.float64).sum(dim=1).cpu().numpy()
    assert np.abs(tot - want).max() <= R.bar(N) * want.max()
    assert bool(torch.isfinite(out).all())
    host = out.cpu().numpy()
    for g in (0, 517, G - 1):
        seg = raw[g * K * N * 2:(g + 1) * K * N * 2].cpu().numpy()
        want_g = R.power_f64(O.unpack_u8iq(seg).astype(np.complex128), N, N, K, None, True, False)
        _check(host[g:g + 1], want_g, N)


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_paths_agree_at_1024(sdr, fmt):
    N, H, K = 1024, 256, 40
    raw, _ = _input(fmt, 30 * K * H, 31)
    w = np.blackman(N).astype(np.float32)
    a = sdr.Psd(N, H, K, window=w, fmt=fmt).process(raw)
    g = sdr.Psd(N, H, K, window=w, fmt=fmt, general=True)
    b = g.process(raw)
    assert g.last_path == 1
    _check(a, b.astype(np.float64), N)


@pytest.mark.parametrize("general", [False, True])
def test_nan_poisons_exactly_its_spectra(sdr, general):
    N, H, K = 1024, 512, 3
    x = gen.complex_noise(40 * K * H, 41)
    pos = 17 * K * H + 100  # in frames j with (j + 1) H - N <= pos < (j + 1) H
    x[pos] = np.nan
    got = sdr.Psd(N, H, K, fmt="c64", general=general).process(x)
    hit = {j // K for j in range(got.shape[0] * K) if (j + 1) * H - N <= pos < (j + 1) * H}
    for g in range(got.shape[0]):
        if g in hit:
            assert np.isnan(got[g]).all(), g
        else:
            assert np.isfinite(got[g]).all(), g


# ---- bit-identity ----------------------------------------------------------------------------------------------------
BIT_CASES = [(1024, 512, 33, False), (1024, 3, 70, False), (1024, 1024, 1, False), (1024, 700, 32, True),
             (1000, 250, 33, False), (64, 48, 100, False)]


def _cuts(n, seed, H, K):
    """ragged cut points: 1-sample calls, calls ending inside a chunk and inside a group, large calls"""
    rng = np.random.default_rng(seed)
    cuts, at = [], 0
    for _ in range(150):  # a run of 1-sample calls at the start
        at += 1
        cuts.append(at)
    while at < n:
        at = min(n, at + int(rng.choice([1, 5, H - 1, H * K // 2 + 3, 32 * H + 1, 3 * H * K + 17])))
        cuts.append(at)
    return cuts


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,H,K,general", BIT_CASES)
def test_blockings_clone_reset_equal_one_call(sdr, fmt, N, H, K, general):
    n = 4 * K * H + 3 * N + 5
    raw, _ = _input(fmt, n, 51)
    per = 2 if fmt == "u8iq" else 1
    one = sdr.Psd(N, H, K, window=np.hanning(N), fmt=fmt, general=general).process(raw)
    assert one.shape[0] == (n // H) // K
    p = sdr.Psd(N, H, K, window=np.hanning(N), fmt=fmt, general=general)
    parts, prev, clone, clone_at = [], 0, None, None
    for c in _cuts(n, N + H + K, H, K):
        parts.append(p.process(raw[per * prev:per * c]))
        prev = c
        if clone is None and c > 2 * K * H + H // 2:  # mid-group
            clone, clone_at = p.clone(), c
    assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
    rest = clone.process(raw[per * clone_at:])
    done = (clone_at // H) // K
    assert np.array_equal(_bits(rest), _bits(one[done:]))
    p.reset()
    assert np.array_equal(_bits(p.process(raw)), _bits(one))


@pytest.mark.parametrize("general", [False, True])
def test_output_too_small_then_retry(sdr, general):
    N, H, K = 1024, 512, 33
    raw, _ = _input("c64", 6 * K * H, 61)
    one = sdr.Psd(N, H, K, fmt="c64", general=general).process(raw)
    torch, dev = _torch()
    st = torch.cuda.current_stream(dev)
    p = sdr.Psd(N, H, K, fmt="c64", general=general, stream=st)
    d_in = torch.from_numpy(raw).to(dev)
    n = raw.size
    G = p.output_count(n)
    out = torch.empty((G, N), dtype=torch.float32, device=dev)
    with pytest.raises(sdr.SdrError):
        p.process_dev(d_in, n, out, G - 1)
    assert p.process_dev(d_in, n, out, G) == G
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(one))


@pytest.mark.parametrize("general", [False, True])
@pytest.mark.parametrize("H", [1024, 512, 8, 3])
def test_unaligned_u8_addresses(sdr, general, H):
    torch, dev = _torch()
    N, K = 1024, 33
    n = 5 * K * H + 2000
    raw = gen.random_u8(2 * n, 71)
    one = sdr.Psd(N, H, K, fmt="u8iq", general=general).process(raw)
    st = torch.cuda.current_stream(dev)
    for off in (2, 6, 14):  # bytes past a 16-byte boundary: element-aligned only
        buf = torch.zeros(2 * n + 64, dtype=torch.uint8, device=dev)
        buf[off:off + 2 * n] = torch.from_numpy(raw).to(dev)
        p = sdr.Psd(N, H, K, fmt="u8iq", general=general, stream=st)
        out = torch.empty((one.shape[0], N), dtype=torch.float32, device=dev)
        base, got, at = buf.data_ptr() + off, 0, 0
        for m in (1001, 3 * H * K + 5, n):  # three calls: every block starts at a different alignment
            m = min(m, n - at)
            got += p.process_dev(base + 2 * at, m, out[got:], one.shape[0] - got)
            at += m
        torch.cuda.synchronize()
        assert got == one.shape[0]
        if not general:
            assert p.last_path == 2
        assert np.array_equal(_bits(out.cpu().numpy()), _bits(one)), off


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
@pytest.mark.parametrize("N,H,K,general", [(1024, 256, 33, False), (1024, 2048, 3, False), (1000, 300, 5, False),
                                           (1024, 256, 33, True)])
def test_shards_concatenate_to_one_stream(sdr, fmt, N, H, K, general):
    """cut on group boundaries; each shard is primed with whole groups covering max(N - H, 0) samples"""
    n_groups = 12
    n = n_groups * K * H
    raw, _ = _input(fmt, n, 81)
    per = 2 if fmt == "u8iq" else 1
    w = np.hanning(N).astype(np.float32)
    one = sdr.Psd(N, H, K, window=w, fmt=fmt, general=general).process(raw)
    prime = -(-max(N - H, 0) // (K * H))  # whole groups
    parts = []
    for g0, g1 in ((0, 4), (4, 9), (9, n_groups)):
        a = max(0, g0 - prime)
        p = sdr.Psd(N, H, K, window=w, fmt=fmt, general=general)
        got = p.process(raw[per * a * K * H: per * g1 * K * H])
        parts.append(got[g0 - a:])
    assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))


def test_power_spectra_over_a_signal(sdr):
    rate, fps, avg = 1024000.0, 2000.0, 8
    iq = gen.tone_noise_u8(300000, rate, 4.0e4, 0.5, 0.05, 8)
    sig = sdr.signal.from_u8iq(rate, iq)
    w = np.hanning(1024).astype(np.float32)
    got = list(sdr.signal.power_spectra(sig, 1024 / rate, fps, avg, window=w, block=12345))
    spectra = np.concatenate([s for _, s in got])
    want = sdr.Psd(1024, 512, avg, window=w, fmt="u8iq").process(iq)
    assert np.array_equal(_bits(spectra), _bits(want))
    labels = got[0][0]
    assert abs(labels[np.argmax(spectra[-1])] - 4.0e4) <= rate / 1024


def test_psd_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "psd_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "PSD MIRROR OK" in r.stdout, r.stdout + r.stderr

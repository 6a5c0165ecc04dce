"""Fast-convolution synthesis bank (sdr_fcsb): every output against f64 truth (zero-stuff, filter, exact 64-bit mixer,
sum, each channel at its own I_k) and against the crate's composition through the CPU oracle; agreement with sdr_duc;
the adjoint identity and the round trip with GPU sdr_fcfb; the round-off bound in terms of ||h_k|| and the block rms;
64-bit stream positions; bit-identity across blockings, clones, resets, retries, strides and block-aligned primed
shards; NaN poisoning of exactly the spanned blocks; draining; spot outputs at 2^28; the C++ mirror."""
import ctypes as C_
import math
import os
import subprocess

import numpy as np
import pytest
from scipy import signal as S

import ddc_ref as R
import duc_ref
import fcfb_ref
import fcsb_ref as Q
import gen
import oracle_lib as O
import pfs_ref
from test_fcsb_host import F_BIG, F_TOP, ROUND_TRIP, ROUND_TRIP_SNR_DB, round_trip_input

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TWO64 = 1 << 64


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _torch():
    import torch
    return torch, torch.device("cuda", 0)


def bar(N):
    return 2 * 1e-5 * math.log2(N)


def _freqs(C, seed):
    return np.random.default_rng(seed + C).uniform(-0.5, 0.5, C)


def _taps(Is, L, per_channel=True):
    """low-pass synthesis taps of gain I_k (cutoff 0.45 / I_k, slightly different per channel), [C, L]"""
    if L == 1:
        return np.array([[float(I)] for I in Is], np.float32)
    rows = [int(I) * gen.lowpass_taps(L, (0.4 + 0.05 * k / len(Is)) / int(I), 1.0) for k, I in enumerate(Is)]
    if not per_channel:
        rows = [rows[0]] * len(Is)
    return np.stack(rows).astype(np.float32)


def _rows(Is, n_time, seed):
    return [gen.complex_noise(n_time // int(I), seed + k) for k, I in enumerate(Is)]


def _incs(bank):
    return [int(v) for v in bank.phase_inc]


def truth_f64(h, rows, incs, Is, first=0):
    """the definition in f64 (fft convolution of each zero-stuffed channel, the exact mixer, the sum)"""
    n = Q.n_time_of(rows, Is)
    out = np.zeros(n, np.complex128)
    for k, (inc, I) in enumerate(zip(incs, Is)):
        s = pfs_ref.zero_stuff(np.asarray(rows[k], np.complex128), int(I))
        hk = np.asarray(R.taps_of(h, k), np.float64)
        u = S.fftconvolve(s, hk)[:n] if hk.size > 1 else s * hk[0]
        out += u * duc_ref.rot_up(R.phases(first, np.arange(n), inc))
    return out


def oracle_f32(h, rows, incs, Is, first=0):
    """the crate's blocks through the CPU oracle: zero-stuff, Fir(h_k) on c64, an f32 mix, the sum in f32"""
    n = Q.n_time_of(rows, Is)
    out = np.zeros(n, np.complex64)
    for k, (inc, I) in enumerate(zip(incs, Is)):
        u = O.Fir(np.asarray(R.taps_of(h, k), np.float32)).apply(
            pfs_ref.zero_stuff(np.asarray(rows[k], np.complex64), int(I)))
        out += (u * duc_ref.rot_up(R.phases(first, np.arange(n), inc)).astype(np.complex64)).astype(np.complex64)
    return out


def _n_time(Is, L, blocks=3, extra=777):
    N, _ = Q.geometry(L, Is)
    Il = Q.lcm_of(Is)
    return -(-(blocks * N + extra) // Il) * Il


CASES = [([8], 255), ([8, 10, 1, 40, 2], 255), ([3, 5, 7], 64), ([1], 1), ([8] * 8, 4095),
         ([8, 8, 16, 16, 32, 32, 64, 64], 4095), ([2] * 256, 64), ([1, 2] * 128, 255), ([10] * 17, 1000),
         ([4, 1], 4095)]


@pytest.mark.parametrize("Is,L", CASES)
def test_fcsb_every_output_against_f64_and_oracle(sdr, Is, L):
    i = CASES.index((Is, L))
    h = _taps(Is, L, per_channel=bool(i % 2))
    n = _n_time(Is, L)
    rows = _rows(Is, n, 40 + i)
    b = sdr.Fcsb(h, _freqs(len(Is), i), 1.0, Is, first_sample=F_BIG)
    N, P = Q.geometry(L, Is)
    assert b.geometry == (N, P)
    assert b.output_count(n) == Q.counts(n, P, Q.off0(F_BIG, Is, P))
    got = b.process(rows)
    assert got.size == Q.counts(n, P, Q.off0(F_BIG, Is, P))
    truth = truth_f64(h, rows, _incs(b), Is, F_BIG)[:got.size]
    assert np.abs(got - truth).max() <= bar(N) * np.abs(truth).max()
    if len(Is) <= 17:
        oracle = oracle_f32(h, rows, _incs(b), Is, F_BIG)[:got.size]
        assert np.abs(got - oracle).max() <= (bar(N) + 1e-5) * np.abs(truth).max()


@pytest.mark.parametrize("I,L,C", [(8, 255, 8), (10, 255, 3), (8, 4095, 8), (1, 64, 2)])
def test_fcsb_equals_duc_when_every_interpolation_is_equal(sdr, I, L, C):
    h = _taps([I] * C, L)
    freqs = _freqs(C, I)
    n = _n_time([I], L)
    y = np.stack(_rows([I] * C, n, 9))
    b = sdr.Fcsb(h, freqs, 1.0, I, first_sample=F_TOP)
    got = b.process(y)
    duc = sdr.Duc(h, freqs, 1.0, I, first_sample=F_TOP).process(y)[:got.size]
    truth = truth_f64(h, list(y), _incs(b), [I] * C, F_TOP)[:got.size]
    N, _ = Q.geometry(L, [I])
    assert np.abs(got - truth).max() <= bar(N) * np.abs(truth).max()
    assert np.abs(got - duc).max() <= (bar(N) + 1e-5) * np.abs(truth).max()


def test_fcsb_adjoint_of_gpu_fcfb(sdr):
    """<v, fcfb(x)> = <fcsb'(v), x>: fcsb' with reversed taps, first_sample F - (L - 1), zero frames appended"""
    Is, L, F = [8, 10, 1, 40], 255, F_BIG
    C = len(Is)
    rng = np.random.default_rng(4)
    h = rng.standard_normal((C, L)).astype(np.float32)
    freqs = _freqs(C, 4)
    Il = Q.lcm_of(Is)
    n = 400 * Il
    x = gen.complex_noise(n, 6)
    fb = sdr.Fcfb(h, freqs, 1.0, Is, "c64", first_sample=F)
    N, _ = fb.geometry
    y = [np.concatenate([a, t])[:n // I] for a, t, I in zip(fb.process(x), fb.process(np.zeros(N, np.complex64)), Is)]
    v = [gen.complex_noise(n // I, 7 + k) for k, I in enumerate(Is)]
    Z = -(-(N + L) // Il) * Il
    sb = sdr.Fcsb(np.ascontiguousarray(h[:, ::-1]), freqs, 1.0, Is, first_sample=(F - (L - 1)) % TWO64)
    xh = sb.process([np.concatenate([vk, np.zeros(Z // I, np.complex64)]) for vk, I in zip(v, Is)])
    assert xh.size >= L - 1 + n
    lhs = sum(np.sum(np.conj(vk.astype(np.complex128)) * yk) for vk, yk in zip(v, y))
    rhs = np.sum(np.conj(xh[L - 1:L - 1 + n].astype(np.complex128)) * x)
    # each side is a sum of terms with relative error <~ bar(N) of the largest: bound incoherently
    scale = math.sqrt(sum(np.sum(np.abs(vk) ** 2) for vk in v) * sum(np.sum(np.abs(yk) ** 2) for yk in y)) + \
        math.sqrt(np.sum(np.abs(xh) ** 2) * np.sum(np.abs(x) ** 2))
    assert abs(lhs - rhs) <= bar(N) * scale


@pytest.mark.parametrize("fmt", ["u8iq", "c64"])
def test_fcfb_fcsb_round_trip_device_resident(sdr, fmt):
    """sdr_fcfb's output rows at its out_stride are sdr_fcsb's input rows at the same in_stride, no host step"""
    torch, dev = _torch()
    Ds, L, nus = ROUND_TRIP["Ds"], ROUND_TRIP["L"], ROUND_TRIP["nus"]
    h, f = Q.kaiser_pairs(Ds, L)
    h, f = h.astype(np.float32), f.astype(np.float32)
    n, F = 820 * 40, F_BIG
    if fmt == "u8iq":
        raw = gen.random_u8(2 * n, 31)
        x = O.unpack_u8iq(raw).astype(np.complex128)
        incs = [R.phase_increment_exact(nu, 1.0) for nu in nus]
    else:
        x, incs = round_trip_input(n, F, nus, ROUND_TRIP["bw"])
        raw = x.astype(np.complex64)
    d = L - 1
    st = torch.cuda.current_stream(dev)
    fb = sdr.Fcfb(h, nus, 1.0, Ds, fmt, first_sample=F, stream=st)
    sb = sdr.Fcsb(f, nus, 1.0, Ds, first_sample=(F - d) % TWO64, stream=st)
    N, P = fb.geometry
    assert sb.geometry == (N, P)
    Il = Q.lcm_of(Ds)
    # analysis: the stream, then N zeros; synthesis: what that released, then zero frames covering N positions
    zeros = np.zeros(2 * N if fmt == "u8iq" else N, np.uint8 if fmt == "u8iq" else np.complex64)
    if fmt == "u8iq":
        zeros[:] = 128
    d_in = torch.from_numpy(np.concatenate([np.ascontiguousarray(raw), zeros])).to(dev)
    cnt = fb.output_count(n + N)
    stride = int(cnt.max()) + 7
    Z = -(-N // Il) * Il
    d_y = torch.zeros((len(Ds), stride + Z), dtype=torch.complex64, device=dev)
    assert list(fb.process_dev(d_in, n + N, d_y, int(cnt.max()), stride + Z)) == list(cnt)
    n_time = int(cnt[0]) * Ds[0]
    assert all(int(c) * D == n_time for c, D in zip(cnt, Ds))
    n_time += Z  # the zero frames after the released rows: already zero in d_y
    out_n = sb.output_count(n_time)
    d_x = torch.empty(out_n, dtype=torch.complex64, device=dev)
    assert sb.process_dev(d_y, n_time, d_x, out_n, stride + Z) == out_n >= n
    torch.cuda.synchronize()
    xr = d_x.cpu().numpy()[:n]
    # the host path gives the same bits
    y_host = [d_y[k, :n_time // D].cpu().numpy() for k, D in enumerate(Ds)]
    host = sdr.Fcsb(f, nus, 1.0, Ds, first_sample=(F - d) % TWO64).process(y_host)[:n]
    assert np.array_equal(_bits(host), _bits(xr))
    # against the f64 cascade
    y64 = fcfb_ref.definition_f64(h.astype(np.float64), x, incs, Ds, F)
    x64 = truth_f64(f.astype(np.float64), [np.concatenate([a, np.zeros(Z // D)]) for a, D in zip(y64, Ds)], incs, Ds,
                    (F - d) % TWO64)[:n]
    ff = max(float(np.linalg.norm(f[k].astype(np.float64))) for k in range(len(Ds)))
    tol = bar(N) * max(np.abs(a).max() for a in y64) * ff * math.sqrt(len(Ds)) + bar(N) * np.abs(x64).max()
    assert np.abs(xr - x64).max() <= tol
    if fmt == "c64":
        ref = x[2 * d:n - d]
        sig = np.mean(np.abs(ref) ** 2)
        snr = 10 * np.log10(sig / np.mean(np.abs(xr[3 * d:] - ref) ** 2))
        snr64 = 10 * np.log10(sig / np.mean(np.abs(x64[3 * d:] - ref) ** 2))
        print("fcfb -> fcsb round trip: %.1f dB (f64 cascade %.1f dB)" % (snr, snr64))
        assert snr64 >= ROUND_TRIP_SNR_DB and snr >= snr64 - 1, (snr, snr64)


@pytest.mark.parametrize("first", [F_BIG, F_TOP, TWO64 - 3])
def test_fcsb_64_bit_stream_positions(sdr, first):
    Is, L = [8, 10, 1, 40], 255
    h = _taps(Is, L)
    n = _n_time(Is, L, 4)
    rows = _rows(Is, n, 31)
    b = sdr.Fcsb(h, _freqs(len(Is), 2), 1.0, Is, first_sample=first)
    got = b.process(rows)
    N, P = b.geometry
    assert got.size == Q.counts(n, P, Q.off0(first, Is, P))
    truth = truth_f64(h, rows, _incs(b), Is, first)[:got.size]
    assert np.abs(got - truth).max() <= bar(N) * np.abs(truth).max()


def test_fcsb_round_off_follows_block_power(sdr):
    """a weak channel 60 dB below a strong one: the synthesis error follows max ||f_k||_2 times the rms of the block's
    zero-stuffed frames summed over channels, |x - x_f64| <= 8 eps log2(N) max||f_k||_2 rms_w, eps = 2^-24 (DESIGN.md
    K12); read back through the analysis bank, the weak channel is still far above that error"""
    Is, L = [8, 8], 1023
    h_a = gen.lowpass_taps(L, 0.4 / 8, 1.0).astype(np.float32)
    f = np.stack([8 * h_a, 8 * h_a])
    nus = [-0.3, 0.1]
    n = 1 << 18
    rng = np.random.default_rng(5)
    weak = (1e-3 * (rng.standard_normal(n // 8) + 1j * rng.standard_normal(n // 8)) / math.sqrt(2)).astype(np.complex64)
    strong = (0.9 * np.exp(2j * np.pi * 0.01 * np.arange(n // 8))).astype(np.complex64)
    b = sdr.Fcsb(f, nus, 1.0, Is)
    N, _ = b.geometry
    got = b.process([weak, strong])
    truth = truth_f64(f, [weak, strong], _incs(b), Is)[:got.size]
    rms_w = math.sqrt(sum(np.mean(np.abs(r.astype(np.complex128)) ** 2) / I for r, I in zip((weak, strong), Is)))
    fn = max(float(np.linalg.norm(f[k].astype(np.float64))) for k in range(2))
    bound = 8 * 2.0 ** -24 * math.log2(N) * fn * rms_w
    err = np.abs(got - truth).max()
    print("round-off %.3g, bound %.3g (%.2f of it)" % (err, bound, err / bound))
    assert err <= bound, (err, bound)
    # read back through the analysis bank (f64): the weak channel's own level is far above the error
    back = fcfb_ref.definition_f64(h_a.astype(np.float64), got.astype(np.complex128), _incs(b)[:1], [8])[0]
    ref = fcfb_ref.definition_f64(h_a.astype(np.float64), truth, _incs(b)[:1], [8])[0]
    assert np.abs(back - ref)[L:].max() <= 0.05 * np.abs(ref[L:]).std()


def _cat_rows(rows, a, e, Is):
    return [r[a // int(I):e // int(I)] for r, I in zip(rows, Is)]


@pytest.mark.parametrize("Is,L,first", [([8, 10, 1, 40, 2], 255, 999), ([8], 4095, 0), ([3, 5], 64, 12345),
                                        ([16, 16, 32], 511, 7)])
def test_fcsb_blocking_clone_reset_are_bit_exact(sdr, Is, L, first):
    h = _taps(Is, L, per_channel=False)
    freqs = _freqs(len(Is), 3)
    b = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=first)
    N, P = b.geometry
    Il = Q.lcm_of(Is)
    n = _n_time(Is, L, 5, 3)
    rows = _rows(Is, n, 5)
    one = b.process(rows)
    b.reset()
    assert np.array_equal(_bits(b.process(rows)), _bits(one))
    # cuts: single-Il calls, calls that end mid-block and on a block end, random ones
    rng = np.random.default_rng(L)
    cuts = {Il, 2 * Il, 3 * Il, P - Il, P, 2 * P + Il} | set((rng.integers(1, n // Il, 9) * Il).tolist())
    cuts = [0] + sorted(c for c in cuts if 0 < c < n) + [n]
    for single in (False, True):
        p = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=first)
        pts = list(range(0, min(n, 3 * P), Il)) + [n] if single else cuts
        parts, clone = [], None
        for a, e in zip(pts[:-1], pts[1:]):
            parts.append(p.process(_cat_rows(rows, a, e, Is)))
            if clone is None and a >= n // 2 and (e + Q.off0(first, Is, P)) % P:
                clone, at, made = p.clone(), e, sum(x.size for x in parts)
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))
        if clone is not None:
            assert np.array_equal(_bits(clone.process(_cat_rows(rows, at, n, Is))), _bits(one[made:]))


def test_fcsb_too_small_output_is_refused_without_state_change(sdr):
    torch, dev = _torch()
    Is, L = [8, 10, 1], 127
    h = _taps(Is, L)
    freqs = _freqs(3, 1)
    Il = Q.lcm_of(Is)
    n = 50 * Il * 10
    rows = _rows(Is, n, 8)
    one = sdr.Fcsb(h, freqs, 1.0, Is).process(rows)
    b = sdr.Fcsb(h, freqs, 1.0, Is)
    first = b.process(_cat_rows(rows, 0, 7 * Il, Is))
    rest = _cat_rows(rows, 7 * Il, n, Is)
    n_rest = n - 7 * Il
    need = b.output_count(n_rest)
    stride = n_rest
    y = np.zeros((3, stride), np.complex64)
    for k, r in enumerate(rest):
        y[k, :r.size] = r
    out = np.empty(need, np.complex64)
    got = C_.c_size_t(7)
    assert sdr.lib().sdr_fcsb_process(b.h, y.ctypes.data, n_rest, stride, out.ctypes.data, need - 1,
                                      C_.byref(got)) == 104
    assert got.value == 0
    d_in = torch.from_numpy(y).to(dev)
    d_out = torch.empty(need, dtype=torch.complex64, device=dev)
    assert sdr.lib().sdr_fcsb_process_dev(b.h, d_in.data_ptr(), n_rest, stride, d_out.data_ptr(), need - 1,
                                          C_.byref(got)) == 104
    # n_time not a multiple of lcm(I_k), and a short row stride
    assert sdr.lib().sdr_fcsb_process(b.h, y.ctypes.data, n_rest - 1, stride, out.ctypes.data, need,
                                      C_.byref(got)) == 100
    assert sdr.lib().sdr_fcsb_process(b.h, y.ctypes.data, n_rest, n_rest - 1, out.ctypes.data, need,
                                      C_.byref(got)) == 100
    assert b.output_count(n_rest) == need
    second = b.process(rest)
    assert np.array_equal(_bits(np.concatenate([first, second])), _bits(one))


@pytest.mark.parametrize("Is,L", [([8, 10, 40], 255), ([1, 2], 1000), ([4], 4095)])
def test_fcsb_odd_strides_and_primed_shards(sdr, Is, L):
    """odd device row strides give the host bits; shards cut on block boundaries of the absolute grid, primed with
    frames covering N - P positions rounded up to Il, first_sample = the halo's first position, give one call's bits"""
    torch, dev = _torch()
    C = len(Is)
    h = _taps(Is, L)
    freqs = _freqs(C, 8)
    first = 3 * Q.lcm_of(Is) + 1  # eps != 0
    N, P = Q.geometry(L, Is)
    Il = Q.lcm_of(Is)
    o0 = Q.off0(first, Is, P)
    n = 12 * P + 5 * Il - o0 % P
    rows = _rows(Is, n, 17)
    one = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=first).process(rows)
    st = torch.cuda.current_stream(dev)
    stride = n // min(Is) + 5
    pad = np.full((C, stride), np.nan, np.complex64)
    for k, r in enumerate(rows):
        pad[k, :r.size] = r
    d_y = torch.from_numpy(pad).to(dev)
    cnt = one.size
    d_out = torch.full((cnt + 3,), float("nan"), dtype=torch.complex64, device=dev)
    assert sdr.Fcsb(h, freqs, 1.0, Is, first_sample=first, stream=st).process_dev(d_y, n, d_out, cnt + 3,
                                                                                    stride) == cnt
    torch.cuda.synchronize()
    out = d_out.cpu().numpy()
    assert np.array_equal(_bits(out[:cnt]), _bits(one)) and np.isnan(out[cnt:]).all()
    halo = -(-(N - P) // Il) * Il
    for world in (2, 3):
        cuts = [0] + [(j * 12 // world) * P - o0 for j in range(1, world)] + [n]
        parts = []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            hlo = max(0, lo - halo)
            b = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=first + hlo)
            parts.append(b.process(_cat_rows(rows, hlo, hi, Is))[lo - hlo:])
        assert np.array_equal(_bits(np.concatenate(parts)), _bits(one))


@pytest.mark.parametrize("Is,L", [([8, 10, 1], 255), ([40], 1000)])
def test_fcsb_nan_poisons_exactly_its_blocks_and_zero_frames_drain(sdr, Is, L):
    h = _taps(Is, L)
    freqs = _freqs(len(Is), 1)
    b = sdr.Fcsb(h, freqs, 1.0, Is, first_sample=5)
    N, P = b.geometry
    Il = Q.lcm_of(Is)
    o0 = Q.off0(5, Is, P)
    n = _n_time(Is, L, 8, 100)
    rows = _rows(Is, n, 2)
    clean = b.clone().process(rows)
    k = len(Is) - 1
    m = rows[k].size // 2 + 3
    rows[k][m] = np.complex64(complex(np.nan, 0.0))
    x = b.process(rows)
    pos = (m + 1) * Is[k] - 1                 # handle position of the NaN frame
    t = np.arange(x.size)
    j = (t + o0) // P                         # block of each output
    span_lo = (j + 1) * P - o0 - N
    hit = (span_lo <= pos) & (pos < span_lo + N)
    assert hit.sum() >= P
    assert np.isnan(x[hit]).all()
    assert np.array_equal(_bits(x[~hit]), _bits(clean[~hit]))
    # drain: zero frames covering N positions (rounded up to Il) bring out every output of the stream
    rows[k][m] = 0
    p = sdr.Fcsb(h, freqs, 1.0, Is)
    Z = -(-N // Il) * Il
    got = np.concatenate([p.process(rows), p.process([np.zeros(Z // I, np.complex64) for I in Is])])
    assert got.size >= n
    truth = truth_f64(h, rows, _incs(p), Is)
    assert np.abs(got[:n] - truth).max() <= bar(N) * np.abs(truth).max()


def test_fcsb_spot_outputs_at_2_28(sdr):
    torch, dev = _torch()
    Is, L = [8, 8, 16, 16, 32, 32, 64, 64], 4095
    h = _taps(Is, L)
    n = 1 << 28
    g = torch.Generator(device=dev).manual_seed(5)
    d_y = torch.randn((len(Is), n // 8), dtype=torch.complex64, device=dev, generator=g)
    st = torch.cuda.current_stream(dev)
    b = sdr.Fcsb(h, _freqs(len(Is), 11), 1.0, Is, first_sample=F_BIG, stream=st)
    N, P = b.geometry
    cnt = b.output_count(n)
    d_out = torch.empty(cnt, dtype=torch.complex64, device=dev)
    assert b.process_dev(d_y, n, d_out, cnt, n // 8) == cnt
    torch.cuda.synchronize()
    assert cnt > n - P
    for t0 in (0, cnt // 3 + 77, cnt - 4096):
        lo = max(0, (t0 - L) // 64 * 64)
        hi = -(-(t0 + 4096) // 64) * 64
        rows = [d_y[k, lo // I:hi // I].cpu().numpy() for k, I in enumerate(Is)]
        truth = truth_f64(h, rows, _incs(b), Is, (F_BIG + lo) % TWO64)[t0 - lo:t0 - lo + 4096]
        got = d_out[t0:t0 + 4096].cpu().numpy()
        assert np.abs(got - truth).max() <= bar(N) * np.abs(truth).max(), t0
    assert bool(torch.isfinite(torch.view_as_real(d_out)).all())
    del d_y, d_out


def test_fcsb_cpp_mirror():
    exe = os.path.join(ROOT, "tests", "cpp", "fcsb_mirror_test")
    lib = os.path.join(ROOT, "unnamed-rust-sdr_b200", "lib")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, exe + ".cpp", "-L" + lib, "-lsdr_b200",
                           "-Wl,-rpath," + lib, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "FCSB MIRROR OK" in r.stdout, r.stdout + r.stderr

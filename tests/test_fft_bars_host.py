"""CPU: where the f64 bars of fft_bars.py come from.  f32 models of the three algorithms behind FftPlan lengths that are
not single-launch powers of two, in numpy / scipy complex64, each at least 3 times inside its bar (worst row of a few
hundred, with and without the plan's f32 1/sqrt(n)) on u8-like, uniform complex and uniform real input, and for
Bluestein on u8-like input with a DC offset that makes the DC bin 5 ... 240 times rms(X64) (u8 noise at n = 2^26 has
55: fft_bars.py), which is what the peak term of its max bar is for:

- direct DFT: fft_naive_kernel's sequential sum, bin k = sum_i x[i] W[i k mod n], W the f32 table of upload_twiddles;
- Bluestein: chirp and b built as fft_plan_init builds them (j^2 mod 2n, f64 angle, rounded once to f32), then
  a = x chirp, A = fft(a), P = conj(A fft(b)), y = fft(P), X = (conj(y) f32(1/m)) chirp, as bluestein_pre / mul / post;
- four-step: fft_huge_launch's N1 x N2 split with the twiddle W_N^(n2 k1) evaluated in f64 and rounded once.

The inner transforms are scipy's, not the kernels'; test_gpu_fft_paths.py holds those to the power-of-two bars, and
test_gpu_fft_general.py holds each whole path on the GPU to the bars below.  A change to a bar must keep this file
passing: the margin is what allows a kernel whose rounding differs from the model's.
"""
import time

import numpy as np
import pytest
import scipy.fft as sf

import fft_bars as B

MARGIN = 3.0


def _inputs(kind, rows, n, seed):
    rng = np.random.default_rng(seed)
    if kind in ("u8", "u8+dc"):
        r = rng.integers(0, 256, (rows, 2 * n)).astype(np.float64)
        x = (r[:, 0::2] - 128.0) / 128.0 + 1j * (r[:, 1::2] - 128.0) / 128.0
        return (x + (0.4 + 0.4j if kind == "u8+dc" else 0.0)).astype(np.complex64)
    if kind == "real":
        return rng.uniform(-1, 1, (rows, n)).astype(np.complex64)
    return (rng.uniform(-1, 1, (rows, n)) + 1j * rng.uniform(-1, 1, (rows, n))).astype(np.complex64)


def _table(n):
    k = np.arange(n, dtype=np.float64)
    c = -2.0 * np.pi / n
    return (np.cos(c * k) + 1j * np.sin(c * k)).astype(np.complex64)


def direct_model(x):
    rows, n = x.shape
    tw = _table(n)
    k = np.arange(n)
    acc = np.zeros((rows, n), np.complex64)
    for i in range(n):
        acc = acc + x[:, i:i + 1] * tw[(i * k) % n][None, :]
    return acc


def bluestein_model(x):
    rows, n = x.shape
    m = B.bluestein_m(n)
    j = np.arange(n, dtype=np.uint64)
    ang = np.pi * ((j * j) % np.uint64(2 * n)).astype(np.float64) / n
    chirp = (np.cos(ang) - 1j * np.sin(ang)).astype(np.complex64)
    w = (np.cos(ang) + 1j * np.sin(ang)).astype(np.complex64)
    b = np.zeros(m, np.complex64)
    b[:n] = w
    b[m - np.arange(1, n)] = w[1:]
    bf = sf.fft(b)
    a = np.zeros((rows, m), np.complex64)
    a[:, :n] = x * chirp
    p = np.conj(sf.fft(a, axis=1) * bf)
    y = sf.fft(p, axis=1)[:, :n]
    return (np.conj(y) * np.float32(1.0 / m)) * chirp


def fourstep_model(x):
    rows, n = x.shape
    l = B.ilog2(n)
    n1, n2 = 1 << (l // 2), 1 << (l - l // 2)
    s = sf.fft(x.reshape(rows, n1, n2).transpose(0, 2, 1), axis=2)  # [n2][k1]
    q = (np.arange(n2, dtype=np.int64)[:, None] * np.arange(n1, dtype=np.int64)[None, :]) % n
    s = (s * np.exp(-2j * np.pi * q / n).astype(np.complex64)).astype(np.complex64)
    s = sf.fft(s.transpose(0, 2, 1), axis=2)  # [k1][k2]
    return s.transpose(0, 2, 1).reshape(rows, n)  # X[k1 + N1 k2]


def per_row(got, x):
    """rms_rel, max_rel and peak of each row (fft_bars.py), against the f64 transform"""
    ref = np.fft.fft(x.astype(np.complex128), axis=1)
    e2 = np.abs(got.astype(np.complex128) - ref) ** 2
    p2 = np.abs(ref) ** 2
    return np.sqrt(e2.sum(1) / p2.sum(1)), np.sqrt(e2.max(1) / p2.mean(1)), np.sqrt(p2.max(1) / p2.mean(1))


# (path, model, [(n, rows)]): a few hundred rows where that is cheap, fewer at the long lengths
CASES = [
    ("direct", direct_model, [(n, 400) for n in (2, 3, 5, 7, 12, 15, 31, 33, 60, 63)]),
    ("bluestein", bluestein_model, [(65, 400), (127, 400), (257, 300), (1000, 300), (4097, 64), (30000, 16),
                                    (40000, 8), (180000, 2)]),
    ("fourstep", fourstep_model, [(1 << 17, 16), (1 << 20, 2)]),
]


@pytest.mark.parametrize("name,model,lengths", CASES, ids=[c[0] for c in CASES])
def test_models_sit_inside_the_bars(name, model, lengths):
    t0 = time.time()
    report = []
    for n, rows in lengths:
        assert B.path(n) == name
        b_rms, b_max, b_peak = B.bars(n)
        norm = np.float32(1.0) / np.sqrt(np.float32(n))
        for kind in ("u8", "uniform", "real") + (("u8+dc",) if name == "bluestein" else ()):
            x = _inputs(kind, rows, n, 7 * n + len(kind))
            got = model(x)
            # the norm flag is one more f32 product: f32(X) f32(1/sqrt n) against the f64 X / sqrt(n)
            for y in (got, (got * norm).astype(np.complex128) * np.sqrt(n)):
                rms, mx, peak = per_row(y, x)
                r = int(np.argmax(mx / (b_max + b_peak * peak)))
                report.append("%s n=%d %s: rms_rel %.2e (bar %.2e)  max_rel %.2e (bar %.2e at peak %.1f)" % (
                    name, n, kind, rms.max(), b_rms, mx[r], b_max + b_peak * peak[r], peak[r]))
                assert rms.max() * MARGIN <= b_rms, report[-1]
                assert mx[r] * MARGIN <= b_max + b_peak * peak[r], report[-1]
    print("\n" + "\n".join(report) + "\n%.1f s" % (time.time() - t0))


def test_path_selection_and_refusals():
    """the lengths fft_plan_init sends down each path, and the ones it refuses"""
    assert [B.path(n) for n in (1, 2, 4, 8, 3, 63, 65)] == ["direct"] * 6 + ["bluestein"]
    assert B.path(16) == B.path(64) == B.path(1 << 16) == "pow2"
    assert B.path(1 << 15, rfft=True) == B.path(1 << 17) == B.path(1 << 27) == "fourstep"
    assert B.path(1 << 28) is None and B.path((1 << 26) + 1) is None
    assert B.path((1 << 26) - 1) == "bluestein" and B.bluestein_m((1 << 26) - 1) == 1 << 27
    assert B.bluestein_m(65) == 256 and B.bluestein_m(1000) == 2048 and B.bluestein_m(40000) == 1 << 17


def test_pow2_bars_are_the_single_launch_files():
    import test_gpu_fft_paths as P
    assert (B.POW2_RMS, B.POW2_MAX) == (P.RMS_BAR, P.MAX_BAR)

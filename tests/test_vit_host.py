"""CPU: the Viterbi decoder bank's reference model (vit_ref) and ABI without a device.  create rejects every invalid
parameter and fails with NO_DEVICE for a valid one; NULL handles give NULL_HANDLE and the lifecycle contract of the
other handles holds; E(T) against a brute-force count over random blockings; the quantiser's edges; the model is
maximum likelihood on short zero-tailed blocks; noiseless codewords decode for every listed code; the metric spread
stays within its bound; the BER of the K = 7 rate-1/2 code sets the bars the GPU tests use; the C++ restatement of the
model equals the numpy model."""
import ctypes as C
import itertools
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
from scipy.special import erfc

import vit_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# BER workload: K = 7, (0o133, 0o171), L = 64, soft values 1 - 2c plus noise at Eb/N0, sigma = 32, zero start and a
# terminated finish, 256 channels of 4096 message bits (6 zero tail bits) per Eb/N0: 1 048 576 bits.  The model's
# result: 4.93e-3 / 3.13e-4 / 1.34e-5 at 2 / 3 / 4 dB (5169 / 328 / 14 errors).  Decoding errors come in bursts, so
# the count varies more between seeds than a Poisson count would: the bank gave 4.02e-4 at 3 dB on the seed of
# test_gpu_vit.py.  The bars sit about 1.4-2x above the model's result, and at 4 dB leave room for a few bursts.
BER_C, BER_M, BER_L, BER_SCALE = 256, 4096, 64, 32.0
BER_BARS = {2.0: 7e-3, 3.0: 6e-4, 4.0: 5e-5}


def uncoded_ber(ebn0_db):
    return 0.5 * erfc(math.sqrt(10 ** (ebn0_db / 10)))


def ber_workload(ebn0_db, C_, seed):
    K, g = R.CODES["k7"]
    rng = np.random.default_rng(seed)
    msg = rng.integers(0, 2, (C_, BER_M)).astype(np.uint8)
    msg[:, -(K - 1):] = 0
    return msg, R.bpsk(R.encode(msg, K, g), ebn0_db, 0.5, rng)


def test_released_count_against_brute_force():
    """E(T) = max(0, 32 floor(T/32) - L) counts the release points 32 j >= L + 32 reached, 32 bits each, over random
    blockings; output_count sums to it"""
    rng = np.random.default_rng(1)
    for L in (32, 64, 96, 512):
        T = 0
        points = 0
        for _ in range(300):
            step = int(rng.integers(0, 90))
            for t in range(T + 1, T + step + 1):
                points += t % 32 == 0 and t >= L + 32
            T += step
            assert R.released(T, L) == 32 * points
        v = R.Vit(7, (0o133, 0o171), L, 1.0, True, C=3)
        v.T[:] = [0, 31, 1000]
        assert list(v.output_count([L + 32, 1, 1])) == [32, 0, 32 * ((1001 // 32) - (1000 // 32))]


def test_quantiser_edges():
    F = np.float32
    x = np.array([0.5, -0.5, 1.5, -1.5, 2.5, 126.5, -126.5, 127.5, -127.5, 1e30, -1e30, np.inf, -np.inf, np.nan, 0.0,
                  -0.0, 0.49999997], F)
    want = [0, 0, 2, -2, 2, 126, -126, 127, -127, 127, -127, 0, 0, 0, 0, 0, 0]
    assert list(R.quantise(x[None], 1.0)[0]) == want
    # a product that overflows f32 saturates; scales per channel; the product rounds in f32 before the tie
    q = R.quantise(np.array([[3e38, -3e38], [0.25, 0.75]], F), np.array([10.0, 2.0], F))
    assert q.tolist() == [[127, -127], [0, 2]]
    assert R.quantise(np.array([[F(0.1)]]), F(5.0))[0, 0] == 0  # fl(0.1 * 5) = 0.5 exactly: ties to even


def _path_cost(x_q, K, gens, msg):
    c = R.encode(msg, K, gens)
    return int(sum(np.where(c[t], 127 + x_q[t], 127 - x_q[t]).sum() for t in range(len(msg))))


@pytest.mark.parametrize("name", sorted(R.CODES))
def test_model_is_maximum_likelihood(name):
    """zero start, a terminated finish and L >= the block: the decoded zero-tailed message's path cost is the minimum
    over all 2^m messages (brute force, m = 12 free bits)"""
    K, g = R.CODES[name]
    n = len(g)
    rng = np.random.default_rng(len(name) + K)
    m_free = 12 if K <= 7 else 10
    m = m_free + K - 1
    msgs = np.array(list(itertools.product([0, 1], repeat=m_free)), np.uint8)
    msgs = np.concatenate([msgs, np.zeros((len(msgs), K - 1), np.uint8)], axis=1)
    codes = R.encode(msgs, K, g).astype(np.int64)                                      # [2^m, m, n]
    for trial in range(4):
        truth = msgs[rng.integers(0, len(msgs))]
        x = R.bpsk(R.encode(truth, K, g), 1.0, 1.0 / n, rng)
        q = R.quantise(x[None], 30.0)[0]                                               # [m, n]
        costs = np.where(codes == 1, 127 + q[None], 127 - q[None]).sum(axis=(1, 2))
        v = R.Vit(K, g, 32, 30.0, True, C=1)
        assert len(v.process(x[None])[0]) == 0
        dec = v.finish(terminated=True)[0]
        assert len(dec) == m
        assert _path_cost(q, K, g, dec) == costs.min(), (name, trial)


@pytest.mark.parametrize("name", sorted(R.CODES))
def test_noiseless_codewords_decode(name):
    K, g = R.CODES[name]
    rng = np.random.default_rng(K)
    for zero_start, L in ((True, 32), (True, 96), (False, 64)):
        msg = rng.integers(0, 2, (3, 700)).astype(np.uint8)
        msg[:, -(K - 1):] = 0
        state = 0 if zero_start else rng.integers(0, 1 << (K - 1), 3)
        x = (1.0 - 2.0 * R.encode(msg, K, g, state)).astype(np.float32)
        v = R.Vit(K, g, L, 50.0, zero_start, C=3)
        b = v.process(x)
        f = v.finish()
        for k in range(3):
            got = np.concatenate([b[k], f[k]])
            assert len(b[k]) == R.released(700, L) and len(got) == 700
            assert np.array_equal(got[K:], msg[k, K:]) and (zero_start is False or np.array_equal(got, msg[k]))


def test_metric_spread_bound():
    """max m - min m <= (2K - 3) 254 n + 1 at every step, on random saturated soft values with erasures"""
    for K, g in ((3, (5, 7)), (5, (0o23, 0o35, 0o33, 0o37)), (7, (0o133, 0o171))):
        n = len(g)
        rng = np.random.default_rng(K)
        x = rng.choice(np.array([-1e3, 1e3, 0.3, np.nan], np.float32), (4, 400, n))
        v = R.Vit(K, g, 32, 1.0, True, C=4)
        worst = 0
        for t in range(400):
            v.process(x[:, t:t + 1])
            worst = max(worst, int((v.m.max(axis=1) - v.m.min(axis=1)).max()))
        assert worst <= R.spread_bound(K, n), (K, worst)


def test_model_ber_sets_the_bars():
    """K = 7 rate 1/2 at 2, 3 and 4 dB over 2^20 bits each within BER_BARS; at 3 dB at least 30x better than uncoded
    BPSK"""
    K, g = R.CODES["k7"]
    for eb, bar in BER_BARS.items():
        msg, x = ber_workload(eb, BER_C, int(eb * 10))
        v = R.Vit(K, g, BER_L, BER_SCALE, True, C=BER_C)
        b = v.process(x)
        f = v.finish()
        out = np.array([np.concatenate([b[k], f[k]]) for k in range(BER_C)])
        ber = (out != msg).mean()
        print("Eb/N0 %.0f dB: BER %.3g (uncoded %.3g)" % (eb, ber, uncoded_ber(eb)))
        assert ber < bar, (eb, ber)
        if eb == 3.0:
            assert uncoded_ber(eb) / ber >= 30


def _cpp_model(tmp):
    exe = os.path.join(tmp, "vit_model")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "vit_model.cpp")])
    return exe


def run_cpp_model(exe, x, K, gens, L, scale, zero_start, tmp):
    src, dst = os.path.join(tmp, "in.f32"), os.path.join(tmp, "out.u8")
    np.ascontiguousarray(x, np.float32).tofile(src)
    r = subprocess.run([exe, str(K), str(L), str(int(zero_start)), repr(float(np.float32(scale)))]
                       + [str(int(v)) for v in gens] + [src, dst], capture_output=True, text=True, check=True)
    return np.fromfile(dst, np.uint8), int(r.stdout.split()[0])


def test_cpp_model_equals_the_numpy_model():
    rng = np.random.default_rng(5)
    with tempfile.TemporaryDirectory() as tmp:
        exe = _cpp_model(tmp)
        for K, g, L, zs in ((3, (5, 7), 32, True), (7, (0o133, 0o171, 0o165), 64, False),
                            (9, (0o561, 0o753), 96, True), (5, (0o23, 0o35, 0o33, 0o37), 32, False)):
            x = (rng.standard_normal((1500, len(g))) * 2).astype(np.float32)
            x[rng.random(x.shape) < 0.02] = np.nan
            x[rng.random(x.shape) < 0.02] = 1e30
            bits, _ = run_cpp_model(exe, x, K, g, L, 20.0, zs, tmp)
            want = R.model(x[None], K, g, L, 20.0, zs)[0]
            assert np.array_equal(bits, want), (K, L)


# ---- the ABI without a device ------------------------------------------------------------------------------------

def _cfg(sdr, K=7, gens=(0o133, 0o171), L=64, scale=(1.0,), C_=4, zero_start=1, n_scales=None):
    F = sdr._ffi
    g = np.ascontiguousarray(gens, np.uint32)
    s = np.ascontiguousarray(scale, np.float32)
    cfg = F.VitConfig(K, g.ctypes.data if g.size else None, g.size, L, s.ctypes.data if s.size else None,
                      s.size if n_scales is None else n_scales, zero_start, C_, 0, None)
    cfg.keep = (g, s)
    return cfg


def test_vit_argument_validation(sdr):
    lib = sdr.lib()
    err = C.c_int(0)
    nan, inf = float("nan"), float("inf")
    assert lib.sdr_vit_create(None, C.byref(err)) is None and err.value == 100
    bad = [_cfg(sdr, K=2, gens=(3, 1)), _cfg(sdr, K=10, gens=(0o1133, 0o171)),       # K out of range
           _cfg(sdr, gens=(0o133,)), _cfg(sdr, gens=(0o133, 0o171, 0o165, 0o117, 0o127)),  # n out of range
           _cfg(sdr, gens=()),                                                     # NULL gens
           _cfg(sdr, gens=(0, 0o171)), _cfg(sdr, gens=(0o133, 128)),               # g = 0, g >= 2^K
           _cfg(sdr, L=0), _cfg(sdr, L=16), _cfg(sdr, L=48), _cfg(sdr, L=544),     # L
           _cfg(sdr, C_=0), _cfg(sdr, C_=65537),                                   # C
           _cfg(sdr, scale=(0.0,)), _cfg(sdr, scale=(-1.0,)), _cfg(sdr, scale=(nan,)), _cfg(sdr, scale=(inf,)),
           _cfg(sdr, scale=(1.0, 1.0)),                                            # n_scales not 1 or C
           _cfg(sdr, scale=(1.0, 1.0, nan, 1.0)),                                  # a per-channel scale NaN
           _cfg(sdr, scale=())]                                                    # NULL scale
    for i, cfg in enumerate(bad):
        err.value = 0
        assert lib.sdr_vit_create(C.byref(cfg), C.byref(err)) is None and err.value == 100, i
    n = np.zeros(4, np.uintp)
    o = np.zeros(4, np.uintp)
    assert lib.sdr_vit_process(None, None, n.ctypes.data, 0, None, 0, o.ctypes.data) == 103
    assert lib.sdr_vit_process_dev(None, None, n.ctypes.data, 0, None, 0, o.ctypes.data) == 103
    assert lib.sdr_vit_output_count(None, n.ctypes.data, o.ctypes.data) == 103
    assert lib.sdr_vit_finish(None, None, 1, None, 0, o.ctypes.data) == 103
    assert lib.sdr_vit_finish_dev(None, None, 1, None, 0, o.ctypes.data) == 103
    assert lib.sdr_vit_reset(None) == 103
    assert lib.sdr_vit_clone(None, C.byref(err)) is None and err.value == 103
    lib.sdr_vit_destroy(None)
    if sdr.device_count() == 0:
        # valid, at the edges: K = 3 and 9, n = 2 and 4, L = 32 and 512, C = 1 and 65536, per-channel scales
        for cfg in [_cfg(sdr, K=3, gens=(5, 7), L=32, C_=1), _cfg(sdr, K=9, gens=(0o557, 0o663, 0o711, 0o777), L=512),
                    _cfg(sdr, C_=65536, zero_start=0), _cfg(sdr, scale=(1.0, 2.0, 3e-30, 3e30)),
                    _cfg(sdr, K=3, gens=(1, 7))]:
            err.value = 0
            assert lib.sdr_vit_create(C.byref(cfg), C.byref(err)) is None and err.value == 102
            assert lib.sdr_vit_create(C.byref(cfg), None) is None


def test_vit_lifecycle_contract(sdr):
    """the contract test_handle_lifecycle_host.py checks for every other handle"""
    lib = sdr.lib()
    err = C.c_int(-1)
    assert lib.sdr_vit_create(None, C.byref(err)) is None and err.value == 100
    assert lib.sdr_vit_create(None, None) is None
    if sdr.device_count() == 0:
        cfg = _cfg(sdr)
        err.value = -1
        assert lib.sdr_vit_create(C.byref(cfg), C.byref(err)) is None and err.value == 102
        assert lib.sdr_vit_create(C.byref(cfg), None) is None
    err.value = -1
    assert lib.sdr_vit_clone(None, C.byref(err)) is None and err.value == 103
    assert lib.sdr_vit_clone(None, None) is None
    assert lib.sdr_vit_reset(None) == 103
    lib.sdr_vit_destroy(None)


def test_vit_without_device_fails_loudly(sdr):
    if sdr.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(sdr.SdrError) as e:
        sdr.Vit(7, (0o133, 0o171), 64, 4.0, n_channels=3)
    assert e.value.code == 102

"""Viterbi decoder bank (sdr_vit) throughput on one GPU: one JSON line per config.

For each config (C, K, n, L): first a fresh handle's first call of 2048 steps per channel is checked against
vit_ref.model (the released bits of the first and last channel, bit for bit), so that a fast wrong answer cannot be
reported; then, on device-resident rows of coded random bits at Eb/N0 = 3 dB (rows larger than the 126 MB L2 from
C = 8 on, and by choice not at C = 1), three alternating rounds of back-to-back process_dev calls continuing the same
stream, with, in the same run:
  - "torch": a batched Viterbi in torch, the add-compare-select as tensor ops over all channels per step and a torch
    traceback every 32 steps, timed over 256 steps;
  - "numpy": the model on the host cores (vit_ref.Vit), timed over 256 steps of at most 64 channels.
Each is timed with CUDA events (the host clock for numpy); the best round counts.  "cycles_per_step" is the call time at
the card's max SM clock over the steps of one channel (channels run side by side).  Bytes are algorithmic: 4 n in
and 1 out per step; "frac_hbm" is that traffic over the call time against 6552.3 GB/s, the HBM rate the rest of the
project quotes as measured peak.  The card's name, power limit and max SM clock are read in the same run.  Last, the
sdr_ddc -> sdr_tsync -> sdr_eq -> sdr_csync -> sdr_vit chain on 2^26 u8 IQ samples at C = 8, with the chain without
sdr_vit timed beside it for the decoder's share.

    python scripts/bench_vit.py [--quick]
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests"), os.path.dirname(__file__)):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_duc import card  # noqa: E402
from bench_pfb import PEAK_GBS, events_ms  # noqa: E402

GENS = {5: (0o23, 0o33), 7: (0o133, 0o171), 9: (0o561, 0o753, 0o711)}
SCALE = 32.0
BASE_STEPS = 256


def coded_rows(torch, dev, C_, S, K, n, seed):
    """soft values of random bits through a random rate-1/n code stream at 3 dB; the code bits come from an LFSR-like
    torch recurrence-free construction: c_j = parity of the K input bits under g_j, computed with shifts"""
    g = torch.Generator(device=dev).manual_seed(seed)
    u = torch.randint(0, 2, (C_, S + K - 1), device=dev, generator=g, dtype=torch.int32)
    gens = GENS[K][:n] if len(GENS[K]) >= n else GENS[K]
    c = []
    for gj in gens:
        acc = torch.zeros((C_, S), dtype=torch.int32, device=dev)
        for i in range(K):  # bit K-1-i of g taps u_{t-i}
            if (gj >> (K - 1 - i)) & 1:
                acc ^= u[:, K - 1 - i:K - 1 - i + S]
        c.append(acc)
    c = torch.stack(c, -1).float()
    sigma = math.sqrt(1.0 / (2.0 * (1.0 / n) * 10 ** 0.3))
    return ((1.0 - 2.0 * c) + sigma * torch.randn((C_, S, n), device=dev, generator=g)).contiguous()


def spot_check(sdr, torch, d_x, K, g, L, C_, st):
    import vit_ref as R
    n0 = min(2048, d_x.shape[1])
    b = sdr.Vit(K, g, L, SCALE, n_channels=C_, stream=st)
    d_y = torch.empty((C_, n0), dtype=torch.uint8, device=d_x.device)
    cnt = b.process_dev(d_x, n0, d_x.shape[1], d_y, n0)
    torch.cuda.synchronize()
    for k in sorted({0, C_ - 1}):
        want = R.model(d_x[k:k + 1, :n0].cpu().numpy(), K, g, L, SCALE, True)[0]
        if cnt[k] != len(want) or not np.array_equal(d_y[k, :cnt[k]].cpu().numpy(), want):
            raise SystemExit("sdr_vit differs from the model on channel %d of (C, K, L) = (%d, %d, %d)" % (k, C_, K, L))
    b.close()


class TorchViterbi:
    """the same decoder as tensor ops: int32 metrics, the ACS over [C, S] per step, a traceback every 32 steps"""

    def __init__(self, torch, dev, C_, K, g, L):
        import vit_ref as R
        self.t, self.K, self.L, self.S = torch, K, L, 1 << (K - 1)
        pred, pat = R.trellis(K, g)
        n = len(g)
        sgn = np.array([[1 if (p >> j) & 1 else -1 for j in range(n)] for p in range(1 << n)], np.float32)
        self.sgn = torch.from_numpy(sgn).to(dev)
        self.p0, self.p1 = [torch.from_numpy(v).to(dev) for v in pred]
        self.c0, self.c1 = [torch.from_numpy(v).to(dev) for v in pat]
        self.m = torch.zeros((C_, self.S), dtype=torch.int32, device=dev)
        self.m[:, 1:] = (K - 1) * 254 * n + 1
        self.dec = torch.zeros((L + 32, C_, self.S), dtype=torch.uint8, device=dev)
        self.T = 0
        self.ar = torch.arange(C_, device=dev)

    def run(self, x):
        t = self.t
        q = t.round(t.clamp(x * SCALE, -127, 127))
        q = t.where(t.isfinite(x), q, t.zeros_like(q))
        cost = (127 * x.shape[2] + q @ self.sgn.T).to(t.int32)  # [C, steps, P]
        bits = []
        for s in range(x.shape[1]):
            cs = cost[:, s]
            a0 = self.m[:, self.p0] + cs[:, self.c0]
            a1 = self.m[:, self.p1] + cs[:, self.c1]
            d = a1 < a0
            self.m = t.where(d, a1, a0)
            self.dec[self.T % (self.L + 32)] = d
            self.T += 1
            if self.T % 32 == 0 and self.T >= self.L + 32:
                st = t.argmin(self.m, 1)
                out = []
                for j in range(self.L + 32):
                    i = self.T - 1 - j
                    if j >= self.L:
                        out.append(st >> (self.K - 2))
                    st = ((st << 1) & (self.S - 1)) | self.dec[i % (self.L + 32), self.ar, st].long()
                bits.append(t.stack(out[::-1], 1).to(t.uint8))
        return bits


def bench_config(sdr, torch, dev, C_, K, n, L, S, calls, name, power, clk):
    import vit_ref as R
    st = torch.cuda.current_stream(dev)
    g = GENS[K][:n]
    d_x = coded_rows(torch, dev, C_, S, K, n, 99 + C_ + K)
    spot_check(sdr, torch, d_x, K, g, L, C_, st)
    bank = sdr.Vit(K, g, L, SCALE, n_channels=C_, stream=st)
    d_y = torch.empty((C_, S), dtype=torch.uint8, device=dev)
    tv = TorchViterbi(torch, dev, C_, K, g, L)
    xs = d_x[:, :BASE_STEPS]

    def call():
        bank.process_dev(d_x, S, S, d_y, S)

    def tcall():
        tv.run(xs)
    call()
    tcall()
    torch.cuda.synchronize()
    t_ms, b_ms = [], []
    for _ in range(3):  # alternate in one run
        t_ms.append(events_ms(torch, st, call, calls))
        b_ms.append(events_ms(torch, st, tcall, 1))
    ms, tms = min(t_ms), min(b_ms)
    ch = min(C_, 64)
    xh = d_x[:ch, :BASE_STEPS].cpu().numpy()
    t0 = time.perf_counter()
    R.model(xh, K, g, L, SCALE, True)
    np_s = time.perf_counter() - t0
    total = C_ * S
    rec = {"bench": "vit", "C": C_, "K": K, "n": n, "L": L, "steps_per_channel": S, "calls": calls,
           "ms_per_call": round(ms, 4), "window_ms": round(ms * calls, 1),
           "gbits_per_s": round(total / (ms * 1e-3) / 1e9, 4),
           "cycles_per_step": round(ms * 1e-3 * clk * 1e6 / S, 1),
           "frac_hbm": round((4 * n + 1) * total / (PEAK_GBS * 1e9) / (ms * 1e-3), 4),
           "torch": {"gbits_per_s": round(C_ * BASE_STEPS / (tms * 1e-3) / 1e9, 6),
                     "bank_speedup": round((tms / BASE_STEPS) / (ms / S), 1)},
           "numpy": {"mbits_per_s": round(ch * BASE_STEPS / np_s / 1e6, 4),
                     "bank_speedup": round((np_s / (ch * BASE_STEPS)) / (ms * 1e-3 / total), 1)},
           "rounds_ms": [round(v, 4) for v in t_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    print(json.dumps(rec), flush=True)
    del d_x, d_y, tv
    torch.cuda.empty_cache()
    return rec


def bench_chain(sdr, torch, dev, n, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tensor path) -> Tsync at 4 frames per symbol (RRC, P = 32) -> Eq (CMA,
    N = 11) -> Csync QPSK -> Vit (K = 7 rate 1/2, L = 64, uniform start), and the same chain without Vit"""
    import gen
    import tsync_ref as TR
    from test_eq_host import EMAX, MU, RADIUS
    C_, D, Ld, P = 8, 8, 255, 32
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0).astype(np.float32)
    h, _ = TR.rrc_taps(4.0, P, 0.35, 8)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    ana = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    tloop = sdr.tsync_loop_design(0.01, 0.707, TR.gardner_slope(0.35), 4.0) + (2.0, 0.01)
    ts = sdr.Tsync(h, P, 4 << 64, tloop, n_channels=C_, stream=st)
    eq = sdr.Eq(11, (4, MU, RADIUS, EMAX, None), n_channels=C_, stream=st)
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, math.sqrt(2.0) * RADIUS, 1 / (2 * math.pi))
    cs = sdr.Csync((4, kp, ki, 2.0 * RADIUS, 0.01), n_channels=C_, stream=st)
    vit = sdr.Vit(7, (0o133, 0o171), 64, 64.0, n_channels=C_, zero_start=False, stream=st)
    cap = int(ts.max_output(nf).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_q = torch.empty_like(d_s)
    d_z = torch.empty_like(d_s)
    ocap = (cap + 35) // 4 * 4  # device rows are 4-byte aligned
    d_b = torch.empty((C_, ocap), dtype=torch.uint8, device=dev)
    out = {}

    def without():
        ana.reset()
        ts.reset()
        eq.reset()
        cs.reset()
        ana.process_dev(d_in, n, d_y, nf)
        out["got"] = ts.process_dev(d_y, nf, nf, d_s, cap, cap)
        eq.process_dev(d_s, out["got"], cap, d_q, cap)
        cs.process_dev(d_q, out["got"], cap, d_z, cap)

    def call():
        without()
        vit.reset()
        vit.process_dev(d_z, out["got"], cap, d_b, ocap)
    call()
    torch.cuda.synchronize()
    c_ms, w_ms = [], []
    for _ in range(2):
        c_ms.append(events_ms(torch, st, call, 2))
        w_ms.append(events_ms(torch, st, without, 2))
    ms, wms = min(c_ms), min(w_ms)
    rec = {"bench": "ddc_tsync_eq_csync_vit_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": Ld,
           "symbols_per_channel": int(out["got"].min()), "ms_per_call": round(ms, 3), "ms_without_vit": round(wms, 3),
           "vit_share": round((ms - wms) / ms, 4), "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 3), "gpu": name,
           "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="fewer steps per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_vit: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    # (C, K, n, L, steps per channel, calls): C S 4 n bytes of input exceed the 126 MB L2 from C = 8 on (268 MB at
    # n = 2).  The one channel at C = 1 is a 4 MB row by choice: a row past L2 would be 2^24 steps, seconds per call on
    # one latency-bound warp pair
    configs = [(1, 7, 2, 64, 1 << 19, 3), (8, 7, 2, 64, 1 << 22, 2), (1024, 7, 2, 64, 1 << 15, 5),
               (16384, 7, 2, 64, 1 << 11, 5), (65536, 7, 2, 64, 1 << 9, 5), (1024, 5, 2, 32, 1 << 15, 5),
               (1024, 9, 2, 128, 1 << 15, 3), (1024, 9, 3, 128, 1 << 15, 3)]
    for C_, K, n, L, S, calls in configs:
        bench_config(sdr, torch, dev, C_, K, n, L, S >> (4 if args.quick else 0), calls, name, power, clk)
    bench_chain(sdr, torch, dev, 1 << (22 if args.quick else 26), name, power)


if __name__ == "__main__":
    main()

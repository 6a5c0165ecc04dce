"""Frame synchronizer bank (sdr_fsync) throughput on one GPU: one JSON line per config.

Configs: C in {1, 8, 1024, 16384, 65536} x Lp in {32, 64, 256}, in two modes:
  - "search": random QPSK with no word present (th_search = 0.9 is never reached), the worst case: every position is
    correlated over Lp taps;
  - "locked": frames of the word and 1024 QPSK payload symbols (F = Lp + 1024), W = 1, after a first call has locked
    every channel; each call holds S = a whole number of frames per channel, so calls continue the same stream.
For each config a fresh handle's first call is first checked against fsync_ref.model on channels 0 and C - 1 (every
payload symbol and record, bit for bit), so that a fast wrong answer cannot be reported.  Then three alternating
rounds of back-to-back process_dev calls (each copies its counts back and synchronises, as the call does for a user)
and, in the same run:
  - "torch": the correlation and energy by conv1d on the real planes (TF32 off), rho in torch, the hits by nonzero and
    the state machine on the host over the hits (a HIT, then one decision per frame at +F), timed with the host clock
    around a synchronised call;
  - "numpy": the model (fsync_ref.Bank) on the host cores over at most 4 channels of at most 65536 symbols.
Rates are G symbols/s of input.  "frac_fp32_issue" (search) is the count of the kernel's hot loop, 12 FP32
instructions per tap and Lp taps per position, over the call time against 148 SMs x 128 lanes x the max SM clock;
"frac_hbm" (locked) is 8 bytes in per symbol and 8 out per payload symbol over the call time against the HBM rate the
project quotes as measured peak.  The card's name, power limit and max SM clock are read in the same run.  Last, the
six-stage chain sdr_ddc -> sdr_tsync -> sdr_eq -> sdr_csync -> sdr_fsync -> sdr_vit at C = 8, timed beside the same
chain with sdr_vit fed straight from sdr_csync.  Its capture is random u8 IQ with no sync word, so sdr_fsync searches
every position and emits nothing: the pair bounds the bank's cost in the chain, it is not a locked steady state.

    python scripts/bench_fsync.py [--quick]
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

PAY = 1024
FP32_PER_TAP = 12
SMS, LANES = 148, 128


def rows(torch, dev, C_, S, Lp, mode, seed):
    """device rows [C, S] complex64 and the word: unit QPSK, and in locked mode the word every F symbols from 0"""
    import fsync_ref as R
    g = torch.Generator(device=dev).manual_seed(seed)
    k = torch.randint(0, 4, (C_, S), device=dev, generator=g)
    ang = (2 * k + 1).float() * (math.pi / 4)
    x = torch.polar(torch.ones_like(ang), ang)
    w = R.word(Lp, np.random.default_rng(seed))
    if mode == "locked":
        F = Lp + PAY
        d_w = torch.from_numpy(w).to(dev)
        for j in range(S // F):
            x[:, j * F:j * F + Lp] = d_w
    return x.contiguous(), w


def params(mode, Lp):
    return (Lp + PAY, 4, 0.9, 0.9, 1, 3, 1) if mode == "search" else (Lp + PAY, 4, 0.5, 0.3, 1, 3, 1)


def spot_check(sdr, torch, d_x, w, prm, C_):
    import fsync_ref as R
    n0 = min(d_x.shape[1], 4 * (len(w) + PAY))
    b = sdr.Fsync(w, prm, n_channels=C_)
    pc, rc = b.max_output(n0)
    cap, rcap = int(pc.max()), int(rc.max())
    d_y = torch.empty((C_, cap), dtype=torch.complex64, device=d_x.device)
    d_r = torch.empty((C_, rcap, 32), dtype=torch.uint8, device=d_x.device)
    got, rgot = b.process_dev(d_x, n0, d_x.shape[1], d_y, cap, cap, d_r, rcap, rcap)
    for k in sorted({0, C_ - 1}):
        pay, rec = R.model([d_x[k, :n0].cpu().numpy()], w, prm)
        gp = d_y[k, :got[k]].cpu().numpy()
        gr = d_r[k].cpu().numpy().reshape(-1).view(R.REC)[:rgot[k]]
        if gp.tobytes() != pay[0].tobytes() or gr.tobytes() != rec[0].tobytes():
            raise SystemExit("sdr_fsync differs from the model on channel %d (C = %d, Lp = %d)" % (k, C_, len(w)))
    b.close()


class TorchFsync:
    """correlation, energy and rho by conv1d in torch; hits to the host; a host state machine over the hits"""

    def __init__(self, torch, dev, w, prm):
        self.t = torch
        p = torch.from_numpy(w).to(dev)
        pr, pi = p.real.float(), p.imag.float()
        self.wc = torch.stack([torch.stack([pr, pi]), torch.stack([-pi, pr])])   # [2 out, 2 in, Lp]
        self.we = torch.ones((1, 2, len(w)), device=dev)
        self.Ep = float((pr * pr + pi * pi).sum())
        self.F, self.ths, self.thc, self.W = prm[0], prm[2], prm[3], prm[6]

    def run(self, x):
        t = self.t
        planes = t.view_as_real(x).permute(0, 2, 1).contiguous()          # [C, 2, S]
        c = t.nn.functional.conv1d(planes, self.wc)                        # [C, 2, S - Lp + 1]
        e = t.nn.functional.conv1d(planes * planes, self.we)[:, 0]
        rho = (c[:, 0] ** 2 + c[:, 1] ** 2) / (e * self.Ep)
        hits = t.nonzero(rho >= min(self.ths, self.thc)).cpu().numpy()
        frames = 0
        state = {}
        for k, s in hits:  # one HIT per channel, then a decision per frame within W of the expected position
            e_ = state.get(k)
            if e_ is None or s > e_ + self.W:
                state[k] = s + self.F
            elif s >= e_ - self.W:
                frames += 1
                state[k] = s + self.F
        return frames


def bench_config(sdr, torch, dev, C_, Lp, mode, S, calls, name, power, clk):
    import fsync_ref as R
    st = torch.cuda.current_stream(dev)
    prm = params(mode, Lp)
    F = Lp + PAY
    if mode == "locked":
        S = max(F, S // F * F)
    d_x, w = rows(torch, dev, C_, S, Lp, mode, 17 + C_ + Lp)
    spot_check(sdr, torch, d_x, w, prm, C_)
    bank = sdr.Fsync(w, prm, n_channels=C_, stream=st)
    pc, rc = bank.max_output(S)
    cap, rcap = int(pc.max()) + F, int(rc.max()) + 4
    d_y = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_r = torch.empty((C_, rcap, 32), dtype=torch.uint8, device=dev)
    out = {}

    def call():
        out["n"] = bank.process_dev(d_x, S, S, d_y, cap, cap, d_r, rcap, rcap)
    call()  # locks every channel in locked mode
    tf = TorchFsync(torch, dev, w, prm)
    tS = min(S, max(F, (1 << 24) // C_ // F * F if mode == "locked" else (1 << 24) // C_))
    xs = d_x[:, :tS]
    tf.run(xs)
    torch.cuda.synchronize()
    t_ms, b_s = [], []
    for _ in range(3):  # alternate in one run
        t_ms.append(events_ms(torch, st, call, calls))
        t0 = time.perf_counter()
        tf.run(xs)
        torch.cuda.synchronize()
        b_s.append(time.perf_counter() - t0)
    ms, ts = min(t_ms), min(b_s)
    ch, ns = min(C_, 4), min(S, 65536)
    xh = [d_x[k, :ns].cpu().numpy() for k in range(ch)]
    t0 = time.perf_counter()
    R.Bank(w, prm, ch).feed(xh)
    np_s = time.perf_counter() - t0
    total = C_ * S
    pay = int(out["n"][0].sum())
    rec = {"bench": "fsync", "mode": mode, "C": C_, "Lp": Lp, "F": F, "symbols_per_channel": S, "calls": calls,
           "ms_per_call": round(ms, 4), "gsym_per_s": round(total / (ms * 1e-3) / 1e9, 4),
           "payload_per_call": pay, "records_per_call": int(out["n"][1].sum()),
           "torch": {"gsym_per_s": round(C_ * tS / ts / 1e9, 5), "bank_speedup": round((ts / (C_ * tS)) /
                                                                                      (ms * 1e-3 / total), 1)},
           "numpy": {"msym_per_s": round(ch * ns / np_s / 1e6, 4),
                     "bank_speedup": round((np_s / (ch * ns)) / (ms * 1e-3 / total), 1)},
           "rounds_ms": [round(v, 4) for v in t_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    if mode == "search":
        rec["frac_fp32_issue"] = round(FP32_PER_TAP * Lp * total / (SMS * LANES * clk * 1e6) / (ms * 1e-3), 4)
    else:
        rec["frac_hbm"] = round((8 * total + 8 * pay) / (PEAK_GBS * 1e9) / (ms * 1e-3), 4)
    bank.close()
    print(json.dumps(rec), flush=True)
    del d_x, d_y, d_r
    torch.cuda.empty_cache()
    return rec


def bench_chain(sdr, torch, dev, n, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255) -> Tsync at 4 frames per symbol (RRC, P = 32) -> Eq (CMA, N = 11) ->
    Csync QPSK -> Fsync (Lp = 64, F = 1088) -> Vit (K = 7 rate 1/2, L = 64, uniform start), and the same chain with Vit
    fed straight from Csync"""
    import fsync_ref as R
    import gen
    import tsync_ref as TR
    from test_eq_host import EMAX, MU, RADIUS
    C_, D, Ld, P, Lp = 8, 8, 255, 32, 64
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
    fs = sdr.Fsync(R.word(Lp, np.random.default_rng(3)), (Lp + PAY, 4, 0.5, 0.3, 1, 3, 2), n_channels=C_, stream=st)
    vit = sdr.Vit(7, (0o133, 0o171), 64, 64.0, n_channels=C_, zero_start=False, stream=st)
    cap = int(ts.max_output(nf).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_q = torch.empty_like(d_s)
    d_z = torch.empty_like(d_s)
    pcap, rcap = (int(v.max()) for v in fs.max_output(cap))
    d_p = torch.empty((C_, pcap), dtype=torch.complex64, device=dev)
    ocap = (max(cap, pcap) + 35) // 4 * 4
    d_b = torch.empty((C_, ocap), dtype=torch.uint8, device=dev)
    out = {}

    def front():
        for x in (ana, ts, eq, cs, vit):
            x.reset()
        ana.process_dev(d_in, n, d_y, nf)
        out["got"] = ts.process_dev(d_y, nf, nf, d_s, cap, cap)
        eq.process_dev(d_s, out["got"], cap, d_q, cap)
        cs.process_dev(d_q, out["got"], cap, d_z, cap)

    def without():
        front()
        vit.process_dev(d_z, out["got"], cap, d_b, ocap)

    def call():
        front()
        fs.reset()
        npay, _ = fs.process_dev(d_z, out["got"], cap, d_p, pcap, pcap)
        vit.process_dev(d_p, npay, pcap, d_b, ocap)
    call()
    without()
    torch.cuda.synchronize()
    c_ms, w_ms = [], []
    for _ in range(2):
        c_ms.append(events_ms(torch, st, call, 2))
        w_ms.append(events_ms(torch, st, without, 2))
    ms, wms = min(c_ms), min(w_ms)
    rec = {"bench": "ddc_tsync_eq_csync_fsync_vit_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D,
           "symbols_per_channel": int(out["got"].min()), "ms_per_call": round(ms, 3),
           "ms_without_fsync": round(wms, 3), "fsync_share": round((ms - wms) / ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 3), "gpu": name, "power_limit": power}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="fewer symbols per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_fsync: no CUDA device (there is no CPU fallback)")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    # about 2^26 symbols per config (512 MB of c64 input, past the 126 MB L2) except at C = 1 (2^20 symbols: one
    # latency-bound warp) and where one channel needs whole frames
    for C_ in (1, 8, 1024, 16384, 65536):
        for Lp in (32, 64, 256):
            for mode in ("search", "locked"):
                S = (1 << 20) if C_ == 1 else max(4 * (Lp + PAY), (1 << 26) // C_)
                if args.quick:
                    S = max(2 * (Lp + PAY), S >> 4)
                bench_config(sdr, torch, dev, C_, Lp, mode, S, 2 if C_ == 1 else 3, name, power, clk)
    bench_chain(sdr, torch, dev, 1 << (22 if args.quick else 26), name, power)


if __name__ == "__main__":
    main()

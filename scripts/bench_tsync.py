"""Symbol timing recovery bank (sdr_tsync) throughput on one GPU: one JSON line per config.

For each config (C, T, P, L): check a fresh handle's first call (symbols near the start and end of the first and last
channel against the f64 interpolant at their exact positions, and the first 8192 positions against the integer
recurrence replayed from the reported errors) so that a fast wrong answer cannot be reported; then alternate, three
rounds, 20 back-to-back process_dev calls (symbols, positions and errors written) on device-resident torch.randn rows
with, in the same run:
  - "arb_open_loop": sdr_arb at step T/2 on the same taps (two interpolants per symbol and no loop), the price of
    closing the loop;
  - "block_rate": what a user composes today, sdr_arb at T/2, a torch Gardner error per channel and call, copied to the
    host, and sdr_arb_set_steps once per call.
Each is timed with CUDA events; the best round counts.  A tsync call returns after its counts are on the host, so its
time includes that synchronisation.  Symbols per channel are clamp(2^24 / C, 2^11, 2^18).  Bytes are algorithmic:
8 per input frame plus 28 per symbol (8 symbol, 16 position, 4 error); FMA per symbol are 6 ceil(L / P) (two chains of
one interpolated coefficient and a complex accumulate per term).  "frac_hbm" is that traffic over the call time against
6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak; "frac_fp32" is the FMA rate against
148 SMs x 128 lanes at the card's max SM clock, read in the same run with the card's name and power limit;
"cycles_per_symbol" is the call time at that clock over the symbols of one channel (channels run side by side, one
thread each).  The last line is the sdr_ddc -> sdr_tsync chain on 2^28 u8 IQ samples (2 rounds of 2 calls: each
channel's 2^23 symbols run in one thread).

    python scripts/bench_tsync.py [--calls 20] [--quick]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests"), os.path.dirname(__file__)):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_duc import card  # noqa: E402
from bench_pfb import PEAK_GBS, events_ms  # noqa: E402

BETA, SPAN = 0.35, 8


def taps_for(L, P):
    """a low-pass prototype at P times the input rate, cutoff 0.45 of the input rate, sum P"""
    import gen
    t = gen.lowpass_taps(L, 0.45 / P, 1.0).astype(np.float64)
    return (P * t / t.sum()).astype(np.float32)


def loop_for(sdr, period):
    kp, ki = sdr.tsync_loop_design(0.01, 0.707, 1.0, period)
    return (kp, ki, 2.0, 0.01)


def spot_check(d_y, d_s, d_p, d_e, h, P, T, loop, got):
    import arb_ref as A
    import tsync_ref as R
    worst = 0.0
    for k in sorted({0, d_y.shape[0] - 1}):
        g = int(got[k])
        n8 = min(g, 8192)
        po = d_p[k, :n8].cpu().numpy().view(np.uint64)
        pos = [(int(a) << 64) | int(b) for a, b in po]
        R.replay(pos, d_e[k, :n8].cpu().numpy(), T, (np.float32(loop[0]), np.float32(loop[1]), np.float32(loop[2]),
                                                      loop[3]), first=0)
        for s0 in (0, max(0, n8 - 512)):
            taus = pos[s0:s0 + 512]
            at = max(0, (taus[0] >> 64) - h.size // P - 2)
            y = d_y[k, at:(taus[-1] >> 64) + 1].cpu().numpy().astype(np.complex128)
            want = A.computed_f64(h.astype(np.float64), P, y, taus, at=at)
            z = d_s[k, s0:s0 + len(taus)].cpu().numpy()
            worst = max(worst, float(np.abs(z - want).max() / np.abs(want).max()))
    if not worst <= 1e-5:
        raise SystemExit("spot symbols differ from f64 truth: %.3g of max|y| > 1e-5" % worst)
    return worst


def bench_config(sdr, torch, dev, C_, period, P, L, calls, quick, name, power, clk):
    import arb_ref as A
    st = torch.cuda.current_stream(dev)
    T = A.step_of(period, 1.0)
    S = min(max((1 << (20 if quick else 24)) // C_, 1 << 11), 1 << (14 if quick else 18))
    n_in = int(S * period) + L // P + 2
    h = taps_for(L, P)
    loop = loop_for(sdr, period)
    g = torch.Generator(device=dev).manual_seed(99 + C_ + L)
    d_y = torch.randn((C_, n_in), dtype=torch.complex64, device=dev, generator=g)
    bank = sdr.Tsync(h, P, T, loop, n_channels=C_, stream=st)
    cap = int(bank.max_output(n_in).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)
    d_p = torch.empty((C_, cap, 2), dtype=torch.int64, device=dev)
    d_e = torch.empty((C_, cap), dtype=torch.float32, device=dev)
    out = {}

    def call():
        bank.reset()
        out["got"] = bank.process_dev(d_y, n_in, n_in, d_s, cap, cap, d_p, d_e)
    call()
    torch.cuda.synchronize()
    err = spot_check(d_y, d_s, d_p, d_e, h, P, T, loop, out["got"])
    # sdr_arb at T / 2: on-time and mid samples of every symbol, open loop
    half = T // 2
    arb = sdr.Arb(h, P, half, n_channels=C_, stream=st)
    acap = int(arb.output_count(n_in).max())
    d_a = torch.empty((C_, acap), dtype=torch.complex64, device=dev)

    def acall():
        arb.reset()
        arb.process_dev(d_y, n_in, n_in, d_a, acap, acap)

    # the block-rate composition: one Gardner error per channel and call from the T/2 outputs, one set_steps per call
    blk = sdr.Arb(h, P, half, n_channels=C_, stream=st)
    kp = float(loop[0])

    def bcall():
        blk.reset()
        blk.process_dev(d_y, n_in, n_in, d_a, acap, acap)
        ns = (acap - 1) // 2
        y = d_a[:, 0:2 * ns + 1:2]
        m = d_a[:, 1:2 * ns:2]
        e = ((y[:, 1:] - y[:, :-1]) * m.conj()).real.clamp(-2.0, 2.0).mean(dim=1).cpu().numpy()
        blk.set_steps([max(1 << 48, int(half - kp / 2 * float(x) * A.ONE)) for x in e])
    bcall()
    torch.cuda.synchronize()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    t_ms, a_ms, b_ms = [], [], []
    for _ in range(3):  # alternate in one run
        t_ms.append(events_ms(torch, st, call, calls))
        a_ms.append(events_ms(torch, st, acall, calls))
        b_ms.append(events_ms(torch, st, bcall, calls))
    ms, ams, bms = min(t_ms), min(a_ms), min(b_ms)
    got = out["got"]
    total = int(got.sum())
    per = float(got.mean())
    nbytes = 8.0 * C_ * n_in + 28.0 * total
    fma = 6.0 * -(-L // P)
    t_hbm = nbytes / (PEAK_GBS * 1e9)
    t_fp32 = total * fma / (148 * 128 * clk * 1e6)
    rec = {"bench": "tsync", "C": C_, "T": T / A.ONE, "phases": P, "taps": L, "symbols": total, "frames": C_ * n_in,
           "calls": calls, "spot_err_rel": err, "ms_per_call": round(ms, 4),
           "gsymbols_per_s": round(total / (ms * 1e-3) / 1e9, 4),
           "gsamples_per_s_in": round(C_ * n_in / (ms * 1e-3) / 1e9, 3),
           "cycles_per_symbol": round(ms * 1e-3 * clk * 1e6 / per, 1), "fma_per_symbol": fma,
           "frac_hbm": round(t_hbm / (ms * 1e-3), 4), "frac_fp32": round(t_fp32 / (ms * 1e-3), 4),
           "arb_open_loop": {"ms_per_call": round(ams, 4), "tsync_over_arb": round(ms / ams, 2)},
           "block_rate": {"ms_per_call": round(bms, 4), "tsync_over_block_rate": round(ms / bms, 2)},
           "rounds_ms": [round(v, 4) for v in t_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    arb.close()
    blk.close()
    print(json.dumps(rec), flush=True)
    del d_y, d_s, d_p, d_e, d_a
    torch.cuda.empty_cache()
    return rec


def bench_chain(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tensor path) -> Tsync at 4 (1 + 37 ppm) frames per symbol, P = 32,
    RRC matched filter (beta 0.35, span 8)"""
    import arb_ref as A
    import gen
    import tsync_ref as R
    C_, D, Ld = 8, 8, 255
    hd = gen.lowpass_taps(Ld, 0.5 / D, 1.0).astype(np.float32)
    period = 4 * (1 + 37e-6)
    T = A.step_of(period, 1.0)
    P = 32
    h, _ = R.rrc_taps(4.0, P, BETA, SPAN)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    ana = sdr.Ddc(hd, freqs, 1.0, D, "u8iq", stream=st)
    ts = sdr.Tsync(h, P, T, loop_for(sdr, period), n_channels=C_, stream=st)
    cap = int(ts.max_output(nf).max())
    d_s = torch.empty((C_, cap), dtype=torch.complex64, device=dev)

    def call():
        ana.reset()
        ts.reset()
        ana.process_dev(d_in, n, d_y, nf)
        ts.process_dev(d_y, nf, nf, d_s, cap, cap)
    call()
    torch.cuda.synchronize()
    assert np.isfinite(d_s[:, 1000:5096].cpu().numpy()).all()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = min(events_ms(torch, st, call, calls) for _ in range(2))
    rec = {"bench": "ddc_tsync_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": Ld, "tsync_T": period,
           "tsync_phases": P, "tsync_taps": int(h.size), "calls": calls, "ms_per_call": round(ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 2), "ddc_path": ana.last_path, "gpu": name,
           "power_limit": power}
    ana.close()
    ts.close()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="fewer symbols per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_tsync: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    calls = max(20, args.calls)
    # (C, T in frames, P, L)
    configs = [(1, 2 * (1 + 37e-6), 64, 1025), (8, 4 * (1 - 50e-6), 64, 2049), (1024, 2 * (1 + 37e-6), 32, 513),
               (16384, 2 * (1 + 37e-6), 32, 513), (1024, 8.25, 32, 2113)]
    for C_, period, P, L in configs:
        bench_config(sdr, torch, dev, C_, period, P, L, calls, args.quick, name, power, clk)
    # 8 channels of 2^25 frames run as 8 sequential loops: 2 rounds of 2 calls
    bench_chain(sdr, torch, dev, 1 << 24 if args.quick else 1 << 28, 2, name, power)


if __name__ == "__main__":
    main()

"""Arbitrary-ratio resampler bank (sdr_arb) throughput on one GPU: one JSON line per config.

For each config: check spot outputs of a fresh handle's first call against the f64 definition at exact positions (so a
fast wrong answer cannot be reported), then alternate, three rounds, 20 back-to-back process_dev calls of the bank on
device-resident rows (torch.randn, 2^26 outputs over all channels) with what a user has without the bank, each timed
with CUDA events; the best round counts.  The alternatives, in the same run:
  - one sdr_src handle per channel (SincMediumQuality, process_dev, ratio 1 / sigma) -- at C = 1024 on the first 8
    channels only, scaled to C and marked "scaled";
  - sdr_rrb where a rational ratio I / D with I = P gives the same taps per output (sigma = 160/128 <-> 128/160).
Bytes per output are algorithmic: 8 sigma of rows in plus 8 out; FMA per output are the chain's 3 ceil(L / P) (one for
the interpolated coefficient, two for the complex accumulate).  "frac_hbm" is that traffic over the call time against
6552.3 GB/s, the HBM rate the rest of the project quotes as measured peak; "frac_fp32" is the FMA rate against
148 SMs x 128 lanes at the card's max SM clock, read in the same run with the card's name and power limit.  The last
line is the sdr_ddc -> sdr_arb chain on 2^28 u8 IQ samples (2.4 MS/s -> 300 kS/s -> 48 kS/s with a 37 ppm clock
correction).

    python scripts/bench_arb.py [--calls 20] [--quick]
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

SRC_CHANNELS = 8  # sdr_src handles timed at large C (the time is scaled to C)


def taps_for(L, P, sigma):
    """a low-pass prototype at P times the input rate, cutoff 0.45 / max(1, sigma) of the input rate, sum P"""
    import gen
    t = gen.lowpass_taps(L, 0.45 / max(1.0, sigma) / P, 1.0).astype(np.float64)
    return (P * t / t.sum()).astype(np.float32)


def spot_check(d_y, d_z, h, P, steps, cnt):
    """outputs near the start, middle and end of the first and last channel against the f64 definition"""
    import arb_ref as A
    worst = 0.0
    L = h.size
    for k in sorted({0, len(steps) - 1}):
        for r0 in (0, int(cnt[k]) // 2 + 5, max(0, int(cnt[k]) - 2048)):
            taus = [r * steps[k] for r in range(r0, min(r0 + 2048, int(cnt[k])))]
            at = max(0, (taus[0] >> 64) - L // P - 2)
            y = d_y[k, at:(taus[-1] >> 64) + 1].cpu().numpy().astype(np.complex128)
            want = A.computed_f64(h.astype(np.float64), P, y, taus, at=at)
            got = d_z[k, r0:r0 + len(taus)].cpu().numpy()
            worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    if not worst <= 1e-5:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|z| > 1e-5" % worst)
    return worst


class PerChannelSrc:
    """one sdr_src handle per channel (SincMediumQuality), fed the channel's row through process_dev until it is used"""

    def __init__(self, sdr, torch, ratios, st):
        self.torch = torch
        self.ratios = ratios
        self.h = [sdr.SampleRate(sdr.ConverterType.SincMediumQuality, 2, stream=st) for _ in ratios]

    def __call__(self, d_y, n, d_out, cap):
        made = []
        for k, (s, ratio) in enumerate(zip(self.h, self.ratios)):
            s.reset()
            used_all, gen_all = 0, 0
            while used_all < n and gen_all < cap:
                used, got = s.process_dev(ratio, d_y[k, used_all:], n - used_all, d_out[k, gen_all:], cap - gen_all)
                used_all += used
                gen_all += got
                if used == 0 and got == 0:
                    break
            made.append(gen_all)
        return made


def bench_config(sdr, torch, dev, label, n_out, C_, sigma_rate, P, L, rrb, calls, name, power, clk):
    import arb_ref as A
    st = torch.cuda.current_stream(dev)
    step = A.step_of(*sigma_rate)
    sigma = step / A.ONE
    steps = [step] * C_
    per = n_out // C_
    n_in = int(per * sigma) + L // P + 2
    h = taps_for(L, P, sigma)
    g = torch.Generator(device=dev).manual_seed(99 + C_ + L)
    d_y = torch.randn((C_, n_in), dtype=torch.complex64, device=dev, generator=g)
    bank = sdr.Arb(h, P, steps, stream=st)
    cnt = bank.output_count(n_in)
    cap = int(cnt.max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)

    def call():
        bank.reset()
        bank.process_dev(d_y, n_in, n_in, d_z, cap, cap)
    call()
    torch.cuda.synchronize()
    err = spot_check(d_y, d_z, h, P, steps, cnt)
    # alternatives: per-channel sdr_src (a subset at large C) and, where one exists, sdr_rrb on the same taps
    nsrc = min(C_, SRC_CHANNELS)
    src = PerChannelSrc(sdr, torch, [1.0 / sigma] * nsrc, st)
    d_s = torch.empty((nsrc, cap + 64), dtype=torch.complex64, device=dev)
    src(d_y, n_in, d_s, cap + 64)
    rb = None
    if rrb is not None:
        I, D = rrb
        assert I == P and D * A.ONE == step * I
        rb = sdr.Rrb(h, I, D, n_channels=C_, stream=st)
        rcap = int(rb.output_count(n_in).max())
        d_r = torch.empty((C_, rcap), dtype=torch.complex64, device=dev)

        def rcall():
            rb.reset()
            rb.process_dev(d_y, n_in, n_in, d_r, rcap, rcap)
    torch.cuda.synchronize()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    bank_ms, src_ms, rrb_ms = [], [], []
    for _ in range(3):  # alternate in one run
        bank_ms.append(events_ms(torch, st, call, calls))
        src_ms.append(events_ms(torch, st, lambda: src(d_y, n_in, d_s, cap + 64), 1))
        if rb is not None:
            rrb_ms.append(events_ms(torch, st, rcall, calls))
    ms = min(bank_ms)
    sms = min(src_ms) * C_ / nsrc
    total = int(cnt.sum())
    gs = total / (ms * 1e-3) / 1e9
    bpo = 8.0 * C_ * n_in / total + 8.0
    fma = 3.0 * -(-L // P)
    t_hbm = total * bpo / (PEAK_GBS * 1e9)
    t_fp32 = total * fma / (148 * 128 * clk * 1e6)
    rec = {"bench": "arb", "config": label, "C": C_, "sigma": sigma, "phases": P, "taps": L, "n_outputs": total,
           "calls": calls, "spot_err_rel": err, "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2),
           "bytes_per_output": round(bpo, 3), "fma_per_output": fma,
           "frac_hbm": round(t_hbm / (ms * 1e-3), 4), "frac_fp32": round(t_fp32 / (ms * 1e-3), 3),
           "bound": "hbm" if t_hbm > t_fp32 else "fp32",
           "sdr_src": {"ms_per_call": round(sms, 3), "ratio": round(sms / ms, 2), "channels_timed": nsrc,
                       "scaled": nsrc < C_},
           "rounds_ms": [round(v, 4) for v in bank_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    if rb is not None:
        rms = min(rrb_ms)
        rec["sdr_rrb"] = {"I": rrb[0], "D": rrb[1], "ms_per_call": round(rms, 4), "ratio": round(rms / ms, 3)}
        rb.close()
    bank.close()
    print(json.dumps(rec), flush=True)
    del d_y, d_z, d_s
    torch.cuda.empty_cache()
    return rec


def bench_chain(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tensor path) -> Arb at 6.25 (1 + 37 ppm), P = 256, L = 8192"""
    import arb_ref as A
    import gen
    C_, D, L = 8, 8, 255
    h = gen.lowpass_taps(L, 0.5 / D, 1.0).astype(np.float32)
    step = A.step_of(6.25 * (1 + 37e-6), 1.0)
    P, La = 256, 8192
    ha = taps_for(La, P, step / A.ONE)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    ana = sdr.Ddc(h, freqs, 1.0, D, "u8iq", stream=st)
    arb = sdr.Arb(ha, P, step, n_channels=C_, stream=st)
    cap = int(arb.output_count(nf).max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)

    def call():
        ana.reset()
        arb.reset()
        ana.process_dev(d_in, n, d_y, nf)
        arb.process_dev(d_y, nf, nf, d_z, cap, cap)
    call()
    torch.cuda.synchronize()
    assert np.isfinite(d_z[:, cap // 2:cap // 2 + 4096].cpu().numpy()).all()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = min(events_ms(torch, st, call, calls) for _ in range(3))
    rec = {"bench": "ddc_arb_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": L,
           "arb_sigma": step / A.ONE, "arb_phases": P, "arb_taps": La, "calls": calls, "ms_per_call": round(ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 2), "ddc_path": ana.last_path, "gpu": name,
           "power_limit": power}
    ana.close()
    arb.close()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="2^20 outputs per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_arb: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 20 if args.quick else 1 << 26
    calls = max(20, args.calls)
    # (label, C, (rate_in, rate_out), P, L, rational twin on the same taps or None)
    configs = [("1024 x 1+37ppm, P 256, L 4096", 1024, (1 + 37e-6, 1.0), 256, 4096, None),
               ("8 x 48000/44100, P 256, L 8192", 8, (48000.0, 44100.0), 256, 8192, None),
               ("8 x 1/4.41, P 128, L 2048", 8, (1.0, 4.41), 128, 2048, None),
               ("1 x 1.000037, P 256, L 8192", 1, (1.000037, 1.0), 256, 8192, None),
               # a rational twin needs P = I, a power of two: sigma = 160/128 against sdr_rrb at 128/160
               ("8 x 160/128, P 128, L 4096", 8, (160.0, 128.0), 128, 4096, (128, 160))]
    for label, C_, rates, P, L, rrb in configs:
        bench_config(sdr, torch, dev, label, big, C_, rates, P, L, rrb, calls, name, power, clk)
    bench_chain(sdr, torch, dev, 1 << 24 if args.quick else 1 << 28, calls, name, power)


if __name__ == "__main__":
    main()

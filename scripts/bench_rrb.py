"""Rational resampler bank (sdr_rrb) throughput on one GPU: one JSON line per config.

For each config: check spot outputs of a fresh handle's first call against the f64 computed form (so a fast wrong
answer cannot be reported), then alternate, three rounds, 20 back-to-back process_dev calls of the bank on
device-resident rows (torch.randn, 2^26 outputs over all channels) with the composition a user would write from the
library -- per channel, zero-stuff in torch and Fir(h_k) on c64 decimating by D_k on its default path, fed in pieces of
at most 2^27 stuffed samples (the Fir handle carries its state across pieces; one multi-channel handle when the
channels share ratio and taps); for I = 1 that is sdr_fir
alone -- each timed with CUDA events; the best round counts.  Bytes per output are algorithmic: 8 D / I of rows in plus
8 out; FMA per output are the chain's 2 ceil(L / I).  "frac_hbm" is that traffic over the call time against 6552.3
GB/s, the HBM rate the rest of the project quotes as measured peak; "frac_fp32" is the FMA rate against 148 SMs x 128
lanes at the card's max SM clock, read in the same run with the card's name and power limit.  The last line is the
sdr_ddc -> sdr_rrb chain on 2^28 u8 IQ samples.

    python scripts/bench_rrb.py [--calls 20] [--quick]
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

PIECE = 1 << 27  # stuffed samples per Fir call in the composition

MIXED = [(1, 5), (4, 25), (2, 25), (3, 4), (147, 160), (75, 64), (147, 8000), (1, 1)]


def taps_for(Is, Ds, L, shared):
    """low-pass rows with cutoff 0.45 / max(I, D) and DC gain I"""
    import gen
    rows = []
    for I, D in (zip(Is[:1], Ds[:1]) if shared else zip(Is, Ds)):
        t = gen.lowpass_taps(L, 0.45 / max(I, D), 1.0)
        rows.append(I * t / t.sum())
    t = np.asarray(rows, np.float32)
    return t[0] if shared else t


class Composition:
    """zero-stuff (torch) and Fir(h) c64 decimating by D on its default path, in pieces of at most PIECE stuffed
    samples: one multi-channel Fir when every channel has the same ratio and taps, else one Fir per channel"""

    def __init__(self, sdr, torch, h, Is, Ds, st):
        self.torch = torch
        C_ = len(Is)
        if h.ndim == 1 and len(set(zip(Is, Ds))) == 1:
            groups = [(list(range(C_)), h, Is[0], Ds[0])]
        else:
            groups = [([k], h if h.ndim == 1 else h[k], Is[k], Ds[k]) for k in range(C_)]
        self.groups = [(ks, I, sdr.Fir(np.ascontiguousarray(hk, np.float32), "c64", decimation=D, n_channels=len(ks),
                                       stream=st)) for ks, hk, I, D in groups]

    def __call__(self, d_y, n_in, d_out):
        torch = self.torch
        cap = d_out.shape[1]
        for ks, I, fir in self.groups:
            fir.reset()
            n_k = int(n_in[ks[0]])
            fpp = max(1, PIECE // (I * len(ks)))  # frames per piece
            rows = d_y[ks[0]:ks[-1] + 1]
            z = torch.zeros((len(ks), fpp * I), dtype=torch.complex64, device=d_y.device) if I > 1 else None
            made = 0
            for a in range(0, n_k, fpp):
                b = min(n_k, a + fpp)
                if I > 1:
                    z[:, I - 1:(b - a) * I:I] = rows[:, a:b]
                    src, stride = z, fpp * I
                else:
                    src, stride = rows[:, a:], d_y.shape[1]
                n = (b - a) * I
                made += fir.process_dev(src, n, d_out[ks[0], made:], fir.output_count(n), stride, cap)
            del z


def spot_check(d_y, d_z, h, Is, Ds, cnt):
    """outputs near the start, middle and end of the first and last channel against the f64 chain"""
    worst = 0.0
    L = h.shape[-1]
    for k in sorted({0, len(Is) - 1}):
        I, D = Is[k], Ds[k]
        hk = (h if h.ndim == 1 else h[k]).astype(np.float64)
        for r0 in (0, int(cnt[k]) // 2 + 5, max(0, int(cnt[k]) - 2048)):
            r = np.arange(r0, min(r0 + 2048, int(cnt[k])))
            q, c = (r + 1) * D // I, (r + 1) * D % I
            f0 = max(0, int(q[0]) - L // I - 2)
            y = d_y[k, f0:int(q[-1]) + 1].cpu().numpy().astype(np.complex128)
            i = np.arange(-(-L // I))
            tap = c[:, None] + i[None, :] * I
            j = q[:, None] - 1 - i[None, :]
            ok = (tap < L) & (j >= 0)
            want = (np.where(ok, hk[np.minimum(tap, L - 1)], 0) *
                    np.where(ok, y[np.clip(j - f0, 0, y.size - 1)], 0)).sum(1)
            got = d_z[k, r0:r0 + r.size].cpu().numpy()
            worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    if not worst <= 1e-5:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|z| > 1e-5" % worst)
    return worst


def bench_config(sdr, torch, dev, label, n_out, Is, Ds, L, shared, calls, name, power, clk):
    st = torch.cuda.current_stream(dev)
    C_ = len(Is)
    per = n_out // C_
    n_in = np.array([-(-per * D // I) for I, D in zip(Is, Ds)], np.int64)  # frames for >= per outputs each
    h = taps_for(Is, Ds, L, shared)
    g = torch.Generator(device=dev).manual_seed(99 + C_ + L)
    stride = int(n_in.max())
    d_y = torch.randn((C_, stride), dtype=torch.complex64, device=dev, generator=g)
    bank = sdr.Rrb(h, Is, Ds, stream=st)
    cnt = bank.output_count(n_in)
    cap = int(cnt.max())
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)

    def call():
        bank.reset()
        bank.process_dev(d_y, n_in, stride, d_z, cap, cap)
    call()
    torch.cuda.synchronize()
    err = spot_check(d_y, d_z, h, Is, Ds, cnt)
    comp = Composition(sdr, torch, h, Is, Ds, st)
    d_ref = torch.zeros_like(d_z)
    comp(d_y, n_in, d_ref)
    torch.cuda.synchronize()
    diff = max(float((d_ref[k, :int(cnt[k])] - d_z[k, :int(cnt[k])]).abs().max() / d_ref[k, :int(cnt[k])].abs().max())
               for k in range(C_))
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    bank_ms, comp_ms = [], []
    for _ in range(3):  # alternate the two in one run
        bank_ms.append(events_ms(torch, st, call, calls))
        comp_ms.append(events_ms(torch, st, lambda: comp(d_y, n_in, d_ref), 1))
    ms, cms = min(bank_ms), min(comp_ms)
    total = int(cnt.sum())
    gs = total / (ms * 1e-3) / 1e9
    bpo = float(sum(8.0 * n for n in n_in) / total + 8.0)
    fma = float(sum(2 * -(-L // I) * int(c) for I, c in zip(Is, cnt)) / total)
    t_hbm = total * bpo / (PEAK_GBS * 1e9)
    t_fp32 = total * fma / (148 * 128 * clk * 1e6)
    rec = {"bench": "rrb", "config": label, "C": C_, "I": Is, "D": Ds, "taps": L, "shared_taps": shared,
           "n_outputs": total, "calls": calls, "spot_err_rel": err, "ms_per_call": round(ms, 4),
           "gsamples_per_s": round(gs, 2), "bytes_per_output": round(bpo, 3), "fma_per_output": round(fma, 2),
           "frac_hbm": round(t_hbm / (ms * 1e-3), 4), "frac_fp32": round(t_fp32 / (ms * 1e-3), 3),
           "bound": "hbm" if t_hbm > t_fp32 else "fp32",
           "composition": {"ms_per_call": round(cms, 3), "max_rel_diff": diff, "ratio": round(cms / ms, 2)},
           "rounds_ms": [round(v, 4) for v in bank_ms], "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    del d_y, d_z, d_ref, comp
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def bench_chain(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Ddc (C = 8, D = 8, L = 255, tcgen05 path) -> Rrb 4/25 (L = 401) on the device"""
    import gen
    C_, D, L = 8, 8, 255
    h = gen.lowpass_taps(L, 0.5 / D, 1.0).astype(np.float32)
    hr = taps_for([4], [25], 401, True)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    ana = sdr.Ddc(h, freqs, 1.0, D, "u8iq", stream=st)
    rb = sdr.Rrb(hr, 4, 25, n_channels=C_, stream=st)
    cap = nf * 4 // 25
    d_z = torch.empty((C_, cap), dtype=torch.complex64, device=dev)

    def call():
        ana.reset()
        rb.reset()
        ana.process_dev(d_in, n, d_y, nf)
        rb.process_dev(d_y, nf, nf, d_z, cap, cap)
    call()
    torch.cuda.synchronize()
    assert np.isfinite(d_z[:, cap // 2:cap // 2 + 4096].cpu().numpy()).all()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = min(events_ms(torch, st, call, calls) for _ in range(3))
    rec = {"bench": "ddc_rrb_chain", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": L, "rrb": "4/25",
           "rrb_taps": 401, "calls": calls, "ms_per_call": round(ms, 4),
           "gsamples_per_s_in": round(n / (ms * 1e-3) / 1e9, 2), "ddc_path": ana.last_path, "gpu": name,
           "power_limit": power}
    ana.close()
    rb.close()
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
        raise SystemExit("bench_rrb: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 20 if args.quick else 1 << 26
    calls = max(20, args.calls)
    configs = [("8 x 1/5, L 255", [1] * 8, [5] * 8, 255, True),
               ("8 x 147/160, L 3529", [147] * 8, [160] * 8, 147 * 24 + 1, True),
               ("1024 x 3/4, L 97", [3] * 1024, [4] * 1024, 97, True),
               ("8 mixed, L 1023", [i for i, _ in MIXED], [d for _, d in MIXED], 1023, False),
               ("1 x 75/64, L 1201", [75], [64], 1201, True)]
    for label, Is, Ds, L, shared in configs:
        bench_config(sdr, torch, dev, label, big, Is, Ds, L, shared, calls, name, power, clk)
    bench_chain(sdr, torch, dev, 1 << 24 if args.quick else 1 << 28, calls, name, power)


if __name__ == "__main__":
    main()

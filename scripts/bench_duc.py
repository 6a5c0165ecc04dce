"""Up-converter bank (sdr_duc) throughput on one GPU: one JSON line per config.

For each config: check spot outputs of a fresh handle's first call against the f64 computed form (so a fast wrong
answer cannot be reported), then alternate, three rounds, 20 back-to-back process_dev calls of the bank on
device-resident rows with the composition a user would write from the library -- per channel, zero-stuff in torch,
Fir(h_k) on c64 (its tcgen05 path), a torch multiply by the NCO rotation computed in chunks from the exact integer
phase, and a sum -- each timed with CUDA events; the best round counts.  Stage times of one call come from a separate
torch.profiler run.  Bytes per output are algorithmic: 8 C / I of rows in plus 8 out; FMA per output are the kernel's
C (2 ceil(L / I) + 8).  "frac_hbm" is that traffic over the call time against 6552.3 GB/s, the HBM rate the rest of
the project quotes as measured peak; "frac_fp32" is the FMA rate against 148 SMs x 128 lanes at the card's max SM
clock, read in the same run with the card's name and power limit.  The last config is the ddc -> duc round trip on
2^28 u8 IQ samples.

    python scripts/bench_duc.py [--calls 20] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unnamed-rust-sdr_b200"), os.path.join(ROOT, "tests"), os.path.dirname(__file__)):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_pfb import PEAK_GBS, events_ms  # noqa: E402

F0 = (1 << 40) + 12345
TWO64 = 1 << 64


def card():
    """name, power limit and max SM clock (MHz) of GPU 0"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, power, clk = [s.strip() for s in out.strip().split(",")[:3]]
        return name, power + " W", float(clk)
    except Exception as e:  # the numbers still stand; say the card could not be read
        return "unknown (%s)" % e, "unknown", float("nan")


def stage_times(torch, fn):
    """per-stage device time (ms) of one call, from torch.profiler kernel / copy records"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    stages = {"duc_kernel": 0.0, "ddc": 0.0, "copy": 0.0, "other": 0.0}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.lower()
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        key = "duc_kernel" if "duc_kernel" in name else "ddc" if "ddc" in name else \
            "copy" if "memcpy" in name else "other"
        stages[key] += us / 1000.0
    return {k: round(v, 4) for k, v in stages.items()}


class Composition:
    """per channel: zero-stuff (torch), Fir(h_k) on c64, times e^{+2 pi i phi_k(F + n) / 2^64} (torch, chunks of
    2^24, exact int64 phase), summed into the output"""

    def __init__(self, sdr, torch, dev, h, incs, I, first, st):
        self.torch, self.I, self.first, self.st = torch, I, first, st
        self.incs = [int(v) for v in incs]
        self.firs = [sdr.Fir(np.ascontiguousarray(h if h.ndim == 1 else h[k], np.float32), "c64", stream=st)
                     for k in range(len(self.incs))]

    def __call__(self, d_y, nf, d_out):
        torch, I = self.torch, self.I
        n = nf * I
        z = torch.zeros(n, dtype=torch.complex64, device=d_y.device)
        u = torch.empty(n, dtype=torch.complex64, device=d_y.device)
        d_out.zero_()
        chunk = 1 << 24
        for k, inc in enumerate(self.incs):
            z[I - 1::I] = d_y[k, :nf]
            fir = self.firs[k]
            fir.reset()
            fir.process_dev(z, n, u, n)
            s_inc = inc - TWO64 if inc >= 1 << 63 else inc
            for a in range(0, n, chunk):
                b = min(n, a + chunk)
                idx = torch.arange(a, b, dtype=torch.int64, device=d_y.device) + (self.first - TWO64 if
                                                                                    self.first >= 1 << 63 else
                                                                                    self.first)
                ph = (idx * s_inc).to(torch.float64) * (2 * np.pi / TWO64)  # int64 product wraps mod 2^64
                rot = torch.polar(torch.ones_like(ph), ph).to(torch.complex64)
                d_out[a:b] += u[a:b] * rot
        del z, u


def spot_check(d_y, d_out, h, incs, I, first, nf):
    import duc_ref as R
    L = h.shape[-1]
    worst = 0.0
    n = nf * I
    for t0 in (0, n // 2 + 5, n - 2048):
        f0 = max(0, t0 // I - L // I - 2)
        y = d_y[:, f0:(t0 + 2048) // I + 1].cpu().numpy()
        want = R.computed_f64(h.astype(np.float64), y, incs, I, (first + f0 * I) % TWO64,
                              outputs=np.arange(t0, t0 + 2048) - f0 * I)
        got = d_out[t0:t0 + 2048].cpu().numpy()
        worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    if not worst <= 1e-5:
        raise SystemExit("spot outputs differ from f64 truth: %.3g of max|x| > 1e-5" % worst)
    return worst


def taps_for(C_, L, I):
    import gen
    return np.stack([I * gen.lowpass_taps(L, (0.45 + 0.05 * k / C_) / I, 1.0) for k in range(C_)]).astype(np.float32)


def bench_config(sdr, torch, dev, n_out, C_, I, L, calls, name, power, clk):
    st = torch.cuda.current_stream(dev)
    nf = n_out // I
    h = taps_for(C_, L, I)
    freqs = np.linspace(-0.4, 0.4, C_)
    g = torch.Generator(device=dev).manual_seed(99 + C_ + I)
    d_y = torch.randn((C_, nf), dtype=torch.complex64, device=dev, generator=g)
    d_out = torch.empty(nf * I, dtype=torch.complex64, device=dev)
    bank = sdr.Duc(h, freqs, 1.0, I, first_sample=F0, stream=st)
    incs = [int(v) for v in bank.phase_inc]
    call = lambda: bank.process_dev(d_y, nf, d_out, nf * I)  # noqa: E731
    assert call() == nf * I
    torch.cuda.synchronize()
    err = spot_check(d_y, d_out, h, incs, I, F0, nf)
    comp = Composition(sdr, torch, dev, h, incs, I, F0, st)
    d_ref = torch.empty_like(d_out)
    comp(d_y, nf, d_ref)
    torch.cuda.synchronize()
    diff = float((d_ref - d_out).abs().max() / d_ref.abs().max())
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    bank_ms, comp_ms = [], []
    for _ in range(3):  # alternate the two in one run
        bank_ms.append(events_ms(torch, st, call, calls))
        comp_ms.append(events_ms(torch, st, lambda: comp(d_y, nf, d_ref), 2))
    ms, cms = min(bank_ms), min(comp_ms)
    gs = nf * I / (ms * 1e-3) / 1e9
    bpo = 8.0 + 8.0 * C_ / I
    fma = C_ * (2 * -(-L // I) + 8)
    rec = {"bench": "duc", "n_outputs": nf * I, "C": C_, "I": I, "taps": L, "calls": calls, "spot_err_rel": err,
           "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2), "bytes_per_output": bpo,
           "fma_per_output": fma, "frac_hbm": round(gs * bpo / PEAK_GBS, 4),
           "frac_fp32": round(gs * 1e9 * fma / (148 * 128 * clk * 1e6), 3),
           "composition": {"ms_per_call": round(cms, 3), "max_rel_diff": diff, "ratio": round(cms / ms, 2)},
           "rounds_ms": [round(v, 4) for v in bank_ms], "stages_ms": stage_times(torch, call),
           "gpu": name, "power_limit": power, "max_sm_clock_mhz": clk}
    bank.close()
    del d_y, d_out, d_ref, comp
    torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)
    return rec


def bench_round_trip(sdr, torch, dev, n, calls, name, power):
    """u8 IQ -> Ddc(h) -> Duc(f = D h) on the device, C = 8, D = I = 8, L = 255"""
    import oracle_lib as O
    import pfs_ref
    C_, D, L = 8, 8, 255
    h = pfs_ref.kaiser_lowpass(L, 0.5 / D, 8.0).astype(np.float32)
    f = (D * h).astype(np.float32)
    freqs = np.linspace(-0.4, 0.4, C_)
    st = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    d_in = torch.randint(0, 256, (2 * n,), dtype=torch.uint8, device=dev, generator=g)
    nf = n // D
    d_y = torch.empty((C_, nf), dtype=torch.complex64, device=dev)
    d_x = torch.empty(n, dtype=torch.complex64, device=dev)
    dl = L - 1
    ana = sdr.Ddc(h, freqs, 1.0, D, "u8iq", first_sample=F0, stream=st)
    syn = sdr.Duc(f, freqs, 1.0, D, first_sample=F0 - dl, stream=st)

    def call():
        ana.process_dev(d_in, n, d_y, nf)
        syn.process_dev(d_y, nf, d_x, n)
    call()
    torch.cuda.synchronize()
    x = O.unpack_u8iq(d_in[2 * (n // 2):2 * (n // 2 + 4096)].cpu().numpy())
    assert np.isfinite(x).all() and np.isfinite(d_x[n // 2:n // 2 + 4096].cpu().numpy()).all()
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    ms = min(events_ms(torch, st, call, calls) for _ in range(3))
    gs = n / (ms * 1e-3) / 1e9
    rec = {"bench": "ddc_duc_round_trip", "fmt": "u8iq", "n_samples": n, "C": C_, "D": D, "taps": L,
           "calls": calls, "ms_per_call": round(ms, 4), "gsamples_per_s": round(gs, 2),
           "ddc_path": ana.last_path, "stages_ms": stage_times(torch, call), "gpu": name, "power_limit": power}
    ana.close()
    syn.close()
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="2^22 outputs per config (a rehearsal, not a measurement)")
    args = ap.parse_args()
    import torch
    import sdr_b200 as sdr
    if not torch.cuda.is_available() or sdr.device_count() < 1:
        raise SystemExit("bench_duc: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    name, power, clk = card()
    big = 1 << 22 if args.quick else 1 << 28
    calls = max(20, args.calls)
    for C_, I, L in [(1, 8, 255), (8, 8, 255), (16, 8, 255), (8, 10, 255), (8, 8, 4095)]:
        bench_config(sdr, torch, dev, big // I * I, C_, I, L, calls, name, power, clk)
    bench_round_trip(sdr, torch, dev, big, calls, name, power)


if __name__ == "__main__":
    main()
